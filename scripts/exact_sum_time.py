"""Cost of exact deposition sums (torj_ctx_set_exact_sum): float and exact mode alternated on the same resident bundles,
in one process. Per workload and mode: the k_trace time (CUDA events around the launch, torj_ctx_last_trace_ms) and the
call time (host clock around torj_bundle_trace + torj_bundle_results, which synchronises), medians over the timed
repeats after one warm-up of each mode. Also records whether repeated float runs changed the profile bits, and checks
that the exact runs never did. The card name and power limit are read in the same run.

    python scripts/exact_sum_time.py [--reps 5] [--out profiles/r05_exact_sum.json]"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
import torj_jl_b200 as tj  # noqa: E402
from torj_jl_b200 import _lib  # noqa: E402


def dp(a):
    return a.ctypes.data_as(_lib.c_dp)


def ip(a):
    return a.ctypes.data_as(_lib.c_ip)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def workloads():
    """(name, plasma arrays kwargs, (pos, dirs, w), beam_id, n_beams, options kwargs, s_max)"""
    pos, dirs, w = bench.beam_bundle("beam64k")
    out = [("beam64k", {}, (pos, dirs, w), None, 1, {}, bench.S_MAX),
           ("beam64k alpha_floor=0", {}, (pos, dirs, w), None, 1, dict(alpha_floor=0.0), bench.S_MAX)]
    P, D, W = zip(*[bench.sweep_beam(b) for b in range(128)])
    bid = np.repeat(np.arange(128, dtype=np.int32), len(W[0]))
    out.append(("sweep1m 1/8 shard, 128 profiles", {}, (np.concatenate(P), np.concatenate(D), np.concatenate(W) / 1024.0),
                bid, 128, {}, bench.S_MAX))
    out.append(("beam 1025", {}, bench.beam_bundle("small"), None, 1, {}, bench.S_MAX))
    N0 = tj.pol_tor_angles_2_vector(np.deg2rad(30.0), 0.0)
    out.append(("warm 46 rays, warp per ray", dict(Te0=10e3),
                tj.launch_peripheral_rays(np.array([2.5, 0.0, 0.4]), N0, 0.0174, 1 / 3.99, 95e9), None, 1,
                dict(absorption_model=1, lanes_per_ray=32), 0.6))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_exact_sum.json"))
    args = ap.parse_args()
    tj.abs_Al_init(bench.N_GL)
    L, ctx = tj.lib(), _lib.context()
    psi = np.linspace(0.0, 1.0, bench.N_PSI)
    rows = []
    for name, pkw, (pos, dirs, w), bid, nb, okw, s_max in workloads():
        pl = tj.Plasma(*tj.solovev_arrays(bench.GRID, bench.GRID, **pkw).values())
        opt = _lib.default_options(**okw)
        n = len(w)
        posT, dirT = np.ascontiguousarray(pos.T), np.ascontiguousarray(dirs.T)
        w = np.ascontiguousarray(w, dtype=np.float64)
        fr, md = np.array([95e9]), np.array([1], dtype=np.int32)
        bh = _lib.c_vp()
        _lib.check(L.torj_bundle_create(ctx, n, dp(posT), dp(dirT), dp(w), dp(fr), ip(md), 0, C.byref(bh)))
        try:
            if bid is not None:
                _lib.check(L.torj_bundle_set_beams(bh, nb, ip(np.ascontiguousarray(bid))))
            prof, dep = np.zeros((nb, len(psi))), np.zeros(nb)
            cnt = _lib.TorjCounters()
            t = {0: [], 1: []}
            k = {0: [], 1: []}
            bits = {0: set(), 1: set()}
            for rep in range(args.reps + 1):
                for mode in (0, 1):
                    _lib.check(L.torj_ctx_set_exact_sum(ctx, mode))
                    _lib.check(L.torj_ctx_sync(ctx))
                    t0 = time.perf_counter()
                    _lib.check(L.torj_bundle_trace(bh, pl.handle(ctx), C.byref(opt), float(s_max), len(psi), dp(psi)))
                    _lib.check(L.torj_bundle_results(bh, dp(prof), dp(dep), None, None, None, None, C.byref(cnt)))
                    t1 = time.perf_counter()
                    ms = C.c_double()
                    _lib.check(L.torj_ctx_last_trace_ms(ctx, C.byref(ms)))
                    bits[mode].add(prof.tobytes() + dep.tobytes())
                    if rep > 0:  # rep 0 warms both modes up
                        t[mode].append((t1 - t0) * 1e3)
                        k[mode].append(ms.value)
        finally:
            L.torj_bundle_destroy(bh)
            _lib.check(L.torj_ctx_set_exact_sum(ctx, 0))
        assert len(bits[1]) == 1, f"{name}: exact-sum profiles changed between runs"
        row = dict(workload=name, n_rays=n, n_beams=nb, n_acc=cnt.n_acc,
                   float_ktrace_ms=float(np.median(k[0])), exact_ktrace_ms=float(np.median(k[1])),
                   float_call_ms=float(np.median(t[0])), exact_call_ms=float(np.median(t[1])),
                   float_ktrace_all=k[0], exact_ktrace_all=k[1], float_call_all=t[0], exact_call_all=t[1],
                   float_distinct_profiles=len(bits[0]), exact_distinct_profiles=len(bits[1]))
        row["ktrace_ratio"] = row["exact_ktrace_ms"] / row["float_ktrace_ms"]
        rows.append(row)
        print(f"{name:36s} k_trace float {row['float_ktrace_ms']:9.2f} ms exact {row['exact_ktrace_ms']:9.2f} ms "
              f"({row['ktrace_ratio']:.3f}x); call {row['float_call_ms']:9.2f} / {row['exact_call_ms']:9.2f} ms; "
              f"distinct float profiles {len(bits[0])}/{args.reps + 1}", flush=True)
    out = dict(card=card(), reps=args.reps, note="medians of the timed repeats; float and exact alternated in one process",
               rows=rows)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print("card:", out["card"])


if __name__ == "__main__":
    main()
