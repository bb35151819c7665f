"""Plasma sets on several GPUs: K beams, one per equilibrium, traced (a) as one torj_trace_plasmas call on one device and
(b) as one torj_multi_trace_plasmas call on 1, 2, 4 and 8 devices, whole beams dealt round-robin (block-cyclic with
block_rays = rays per beam). 257 x 257 grid, s_max = 1 m, 1 000 psi levels; K in {32, 128}; the 1 025-ray beam
(N_rings = 7, min_azimuthal_points = 20) and the 5 165-ray beam (21, 11). The plasmas differ in density, temperature and
B0 and are built on the device (build="device", the constructor torj_multi uses). Device counts above the visible GPUs
are reported as not measured.
  python scripts/multi_plasma_set_time.py OUT.json
Wall: host clock around the call (gather, upload, trace, reduction, results copied back: it synchronises). Device: the
k_trace time of the call, the largest over the devices (torj_multi_last_trace_ms / torj_ctx_last_trace_ms). Each is the
median of `REPS` calls after a warm-up call. Construction: host clock around making the K per-device copies of the set
(K x N_dev device builds), once per device count."""
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
DEVICES = (1, 2, 4, 8)


def plasmas(K):
    out = []
    for k in range(K):
        q = k / max(K - 1, 1)
        a = tj.solovev_arrays(257, 257, B0=2.0 + 0.1 * q, ne0=3.0e19 * (0.3 + 0.9 * q), Te0=4.0e3 * (0.8 + 0.6 * q))
        out.append(tj.Plasma(*a.values(), build="device"))
    return out


def timed(fn):
    fn()
    walls, devs, res = [], [], None
    for _ in range(REPS):
        t0 = time.perf_counter()
        res = fn()
        walls.append(1e3 * (time.perf_counter() - t0))
        devs.append(res[1])
    return float(np.median(walls)), float(np.median(devs)), res[0]


def ctx_ms():
    t = C.c_double()
    _lib.check(tj.lib().torj_ctx_last_trace_ms(_lib.context(), C.byref(t)))
    return t.value


def multi_ms(mg):
    t, worst = C.c_double(), 0.0
    for d in range(mg.n_devices):
        _lib.check(tj.lib().torj_multi_last_trace_ms(mg.h, d, C.byref(t)))
        worst = max(worst, t.value)
    return worst


def main(out):
    import torch

    visible = torch.cuda.device_count()
    tj.abs_Al_init(24)
    info = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()
    x0 = np.array([2.5, 0.0, 0.4])
    N0 = tj.pol_tor_angles_2_vector(np.deg2rad(30.0), 0.0)
    beams = {"1025": tj.launch_peripheral_rays(x0, N0, 0.0174, 1 / 3.99, F, N_rings=7, min_azimuthal_points=20),
             "5165": tj.launch_peripheral_rays(x0, N0, 0.0174, 1 / 3.99, F, N_rings=21, min_azimuthal_points=11)}
    pls_all = plasmas(128)
    ctx = _lib.context()
    t0 = time.perf_counter()
    for p in pls_all:
        p.handle(ctx)
    tj.lib().torj_ctx_sync(ctx)
    build_single_ms = 1e3 * (time.perf_counter() - t0)
    rows = []
    for K in (32, 128):
        pls = pls_all[:K]
        for bname, (pos, dirs, w) in beams.items():
            n = len(w)
            P, D, W = np.tile(pos, (K, 1)), np.tile(dirs, (K, 1)), np.tile(w, K)
            B = np.repeat(np.arange(K, dtype=np.int32), n)
            bp = np.arange(K, dtype=np.int32)

            def single():
                return tj.trace_bundle(pls, P, D, W, F, 1, S_MAX, PSI, beam_id=B, n_beams=K, beam_plasma=bp), ctx_ms()

            w1, d1, r1 = timed(single)
            row = dict(beam_rays=n, K=K, rays=K * n, single_wall_ms=w1, single_trace_ms=d1,
                       single_steps=r1["counters"]["n_acc"], multi={})
            print(json.dumps(dict(row, multi=None)), flush=True)
            for nd in DEVICES:
                if nd > visible:
                    row["multi"][str(nd)] = f"not measured ({visible} GPU visible)"
                    continue
                mg = tj.MultiGPU(nd)
                try:
                    mg.abs_Al_init(24)
                    t0 = time.perf_counter()
                    for p in pls:
                        mg._plasma(p)
                    build_ms = 1e3 * (time.perf_counter() - t0)
                    mg.configure("block_cyclic", n)

                    def multi():
                        r = mg.trace_bundle(pls, P, D, W, F, 1, S_MAX, PSI, beam_id=B, n_beams=K, beam_plasma=bp)
                        return r, multi_ms(mg)

                    wm, dm, rm = timed(multi)
                    assert (rm["status"] == r1["status"]).all()
                    dep_rel = float(np.abs(rm["deposited_power"] - r1["deposited_power"]).max() / r1["deposited_power"].max())
                    assert dep_rel < 1e-8, dep_rel
                    m = dict(wall_ms=wm, trace_ms=dm, build_mplasmas_ms=build_ms, speedup_wall_vs_single=w1 / wm,
                             speedup_trace_vs_single=d1 / dm, used_nccl=mg.used_nccl, max_rel_deposited_vs_single=dep_rel,
                             steps=rm["counters"]["n_acc"])
                    row["multi"][str(nd)] = m
                    print(json.dumps(dict(K=K, beam_rays=n, devices=nd, **m)), flush=True)
                finally:
                    mg.close()
            rows.append(row)
    res = dict(gpu=info, visible_gpus=visible, torch_device=torch.cuda.get_device_name(0), grid="257x257", s_max=S_MAX,
               n_psi=len(PSI), reps=REPS, build_128_plasmas_single_device_ms=build_single_ms, rows=rows)
    with open(out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(f"gpu: {info} (visible: {visible})")
    print(f"{'beam':>5} {'K':>4} {'rays':>7} | {'1 dev set ms':>12} {'trace':>8} | {'N':>2} {'multi ms':>9} {'trace':>8} "
          f"{'build':>8} | {'x wall':>6} {'x trace':>7}")
    for r in rows:
        for nd, m in r["multi"].items():
            if isinstance(m, str):
                print(f"{r['beam_rays']:>5} {r['K']:>4} {r['rays']:>7} | {r['single_wall_ms']:>12.1f} {r['single_trace_ms']:>8.1f} "
                      f"| {nd:>2} {m}")
                continue
            print(f"{r['beam_rays']:>5} {r['K']:>4} {r['rays']:>7} | {r['single_wall_ms']:>12.1f} {r['single_trace_ms']:>8.1f} | "
                  f"{nd:>2} {m['wall_ms']:>9.1f} {m['trace_ms']:>8.1f} {m['build_mplasmas_ms']:>8.0f} | "
                  f"{m['speedup_wall_vs_single']:>6.2f} {m['speedup_trace_vs_single']:>7.2f}")


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else "multi_plasma_set_time.json")
