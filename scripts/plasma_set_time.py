"""Plasma sets on one GPU: K beams, one per equilibrium, traced (a) as K sequential torj_trace calls, (b) as one
torj_trace_plasmas call, (c) as the same K beams in ONE plasma via beam ids (isolates the per-ray table base and the lost
sharing of table rows between the plasmas). 257 x 257 grid; K in {1, 8, 32, 128}; the reference's default 46-ray beam
(N_rings = 3, min_azimuthal_points = 5) and the 1 025-ray beam (7, 20). The plasmas differ in density, temperature and B0.
  python scripts/plasma_set_time.py OUT.json
Wall: host clock around the one-shot call (upload, trace, results copied back: it synchronises); device: the sum of
torj_ctx_last_trace_ms of the call(s); each the median of `REPS` after a warm-up call."""
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torj_jl_b200 as tj  # noqa: E402
from torj_jl_b200 import _lib  # noqa: E402

REPS = 3
PSI = np.linspace(0.0, 1.0, 1000)
F, S_MAX = 95e9, 1.0


def plasmas(K):
    out = []
    for k in range(K):
        q = k / max(K - 1, 1)
        a = tj.solovev_arrays(257, 257, B0=2.0 + 0.1 * q, ne0=3.0e19 * (0.3 + 0.9 * q), Te0=4.0e3 * (0.8 + 0.6 * q))
        out.append(tj.Plasma(*a.values()))
    return out


def timed(fn):
    L, ctx = tj.lib(), _lib.context()
    fn()
    walls, devs, res = [], [], None
    for _ in range(REPS):
        t0 = time.perf_counter()
        res, dev = fn()
        walls.append(1e3 * (time.perf_counter() - t0))
        devs.append(dev)
    return float(np.median(walls)), float(np.median(devs)), res


def last_ms():
    t = C.c_double()
    _lib.check(tj.lib().torj_ctx_last_trace_ms(_lib.context(), C.byref(t)))
    return t.value


def main(out):
    tj.abs_Al_init(24)
    info = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()
    x0 = np.array([2.5, 0.0, 0.4])
    N0 = tj.pol_tor_angles_2_vector(np.deg2rad(30.0), 0.0)
    beams = {"46": tj.launch_peripheral_rays(x0, N0, 0.0174, 1 / 3.99, F),
             "1025": tj.launch_peripheral_rays(x0, N0, 0.0174, 1 / 3.99, F, N_rings=7, min_azimuthal_points=20)}
    pls_all = plasmas(128)
    rows = []
    for bname, (pos, dirs, w) in beams.items():
        n = len(w)
        for K in (1, 8, 32, 128):
            pls = pls_all[:K] if K > 1 else pls_all[:1]
            P, D, W = np.tile(pos, (K, 1)), np.tile(dirs, (K, 1)), np.tile(w, K)
            B = np.repeat(np.arange(K, dtype=np.int32), n) if K > 1 else None

            def seq():
                rs, dev = [], 0.0
                for p in pls:
                    rs.append(tj.trace_bundle(p, pos, dirs, w, F, 1, S_MAX, PSI))
                    dev += last_ms()
                return rs, dev

            def one_call():
                r = tj.trace_bundle(pls, P, D, W, F, 1, S_MAX, PSI, beam_id=B, n_beams=K, beam_plasma=np.arange(K))
                return r, last_ms()

            def one_plasma():
                r = tj.trace_bundle(pls[0], P, D, W, F, 1, S_MAX, PSI, beam_id=B, n_beams=K)
                return r, last_ms()

            wa, da, ra = timed(seq)
            wb, db, rb = timed(one_call)
            wc, dc, rc = timed(one_plasma)
            steps_a = sum(r["counters"]["n_acc"] for r in ra)
            steps_b, steps_c = rb["counters"]["n_acc"], rc["counters"]["n_acc"]
            assert steps_a == steps_b, (steps_a, steps_b)
            row = dict(beam_rays=n, K=K, rays=K * n,
                       a_seq_wall_ms=wa, a_seq_trace_ms=da, b_set_wall_ms=wb, b_set_trace_ms=db,
                       c_oneplasma_wall_ms=wc, c_oneplasma_trace_ms=dc,
                       ratio_a_over_b_wall=wa / wb, ratio_c_over_b_trace=dc / db,
                       b_ray_steps_per_s=steps_b / (wb * 1e-3), a_ray_steps_per_s=steps_a / (wa * 1e-3),
                       c_ray_steps_per_s=steps_c / (wc * 1e-3))
            rows.append(row)
            print(json.dumps(row), flush=True)
    res = dict(gpu=info, torch_device=__import__("torch").cuda.get_device_name(0), grid="257x257", s_max=S_MAX,
               n_psi=len(PSI), reps=REPS, rows=rows)
    with open(out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(f"gpu: {info}")
    print(f"{'beam':>5} {'K':>4} {'rays':>7} | {'(a) seq ms':>10} {'dev':>8} | {'(b) set ms':>10} {'dev':>8} | {'(c) 1pl ms':>10} "
          f"{'dev':>8} | {'a/b':>6} {'c/b dev':>7} | {'(b) steps/s':>11}")
    for r in rows:
        print(f"{r['beam_rays']:>5} {r['K']:>4} {r['rays']:>7} | {r['a_seq_wall_ms']:>10.1f} {r['a_seq_trace_ms']:>8.1f} | "
              f"{r['b_set_wall_ms']:>10.1f} {r['b_set_trace_ms']:>8.1f} | {r['c_oneplasma_wall_ms']:>10.1f} "
              f"{r['c_oneplasma_trace_ms']:>8.1f} | {r['ratio_a_over_b_wall']:>6.2f} {r['ratio_c_over_b_trace']:>7.3f} | "
              f"{r['b_ray_steps_per_s']:>11.3e}")


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else "plasma_set_time.json")
