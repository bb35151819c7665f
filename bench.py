#!/usr/bin/env python
"""Headline benchmark of the TorJ ray-tracing hot path (BASELINE.json: ray-steps/s & rays/s of an EC beam bundle).

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (torchrun for N>1, one rank per GPU)
  python bench.py --impl reference --gpus N --steps K ...  # CPU arm: the oracle port on all host cores (the Julia
                                                           # reference itself cannot run here: no Julia, SURVEY.md F2)
  python bench.py --impl multi --gpus N ...                # ONE process driving N devices through torj_multi_trace (what a
                                                           # Julia session binds): host buffers in, NCCL all-reduce inside

A "step" = one pass of the hot path over one bundle. Workloads (--workload; the default depends on N):
  beam64k  BASELINE.json configs[2]: 65 543-ray Gaussian EC beam (N_rings=66, min_az=14), 257x257 Solov'ev equilibrium,
           s_max = 1 m, 1000 psi bins, X-mode 95 GHz. Default at N = 1 (the configuration the metric is quoted on).
  sweep1m  configs[3]: 32 x 32 launcher angles x 1 025-ray beams = 1 049 600 rays, STRONG scaling: the 1 024 beams are
           dealt round-robin over the ranks, one NCCL all-reduce of [dP_dV | deposited | sum w]. Default at N > 1; at
           N = 1 the default run appends a short sweep1m measurement (`strong_scaling_n1`) as the anchor of that curve.
  small    configs[1]: one 1 025-ray beam (a warp per ray).
  config5  configs[4]: 2 launchers x {110, 170} GHz x T_e0 in {10, 15, 25} keV x --c5-angles steering angles x 1 025-ray
           beams with the warm-plasma absorption model (reference src/general_absorption.jl).
Every GPU line carries, outside the timed region, a parity check against the CPU oracle and the GPU time with
alpha_floor = 0 (`exact_ms_per_step`); the CPU arm reports the oracle both exact and with the same work-saving rules.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

GRID, N_PSI, N_GL, S_MAX = 257, 1000, 24, 1.0
# config5: the beams of a scan differ in cost by frequency and temperature (whole beams per rank left the 170 GHz ranks idle while
# the 110 GHz ranks worked: 0.11 of peak on 8 GPUs against 0.16 on one); rays of one beam cost the same, so warp-sized blocks of
# every beam go round the ranks. One profile row per beam on every rank, summed by the same all-reduce.
C5_BLOCK = 32
WORKLOADS = {
    "beam64k": dict(name="config3_64k_ray_beam", n_rays=65543, N_rings=66, min_az=14, f=95e9, mode=1, model=0, scaling="weak"),
    "small": dict(name="config2_1k_ray_beam", n_rays=1025, N_rings=7, min_az=20, f=95e9, mode=1, model=0, scaling="weak"),
    "sweep1m": dict(name="config4_1M_ray_angle_sweep", n_rays=1049600, N_rings=7, min_az=20, f=95e9, mode=1, model=0, scaling="strong"),
    "config5": dict(name="config5_warm_multi_launcher_scan", N_rings=7, min_az=20, model=1, scaling="strong"),
}
# algorithmic FP64 flops per unit (SURVEY.md §8(d); add/mul = 1, FMA = 2, div/sqrt/exp/Bessel call = 1: a lower bound)
F_RHS, F_ALPHA, F_HARM, F_RK_TSIT5, F_DEP = 660.0, 105.0, 1540.0, 440.0, 100.0
# warm model: SURVEY.md §8(d) "add ~0.42 Mflop per alpha call" = 501 nodes x 7 resonance indices x 120 flops; the counter
# n_harm counts resonance indices integrated; 3 000 for the anti-Hermitian part, tensor assembly and fixed-point iteration
F_WARM_N, F_WARM_SOLVE = 501.0 * 120.0, 3000.0


def algorithmic_flops(c, model=0):
    base = F_RHS * c["n_rhs"] + (F_RK_TSIT5 + F_DEP) * c["n_acc"]
    if model == 1:
        return base + F_WARM_N * c["n_harm"] + F_WARM_SOLVE * c["n_harm"] / 7.0
    return base + F_ALPHA * c["n_alpha"] + F_HARM * c["n_harm"]


def make_config(wl, args):
    """The `config` object of the JSON line: the SAME for the GPU arm and the CPU arm (the driver compares them)."""
    w = WORKLOADS[wl]
    cfg = {"workload": w["name"], "grid": f"{GRID}x{GRID}", "s_max": S_MAX, "n_psi": N_PSI, "scheme": "Tsit5",
           "absorption_model": "warm (general_absorption.jl)" if w["model"] else "albajar (absorption.jl)",
           "l2": "compute-bound kernel: tables 4.8 MB L2-resident by design, ray state re-read from HBM each step; no flush needed"}
    if wl == "config5":
        cfg.update(n_rays=12 * args.c5_angles * 1025, launchers=2, f=[110e9, 170e9], Te0_keV=[10, 15, 25], angles=args.c5_angles, mode=1)
    else:
        cfg.update(n_rays=w["n_rays"], f=w["f"], mode=w["mode"])
    return cfg


# ---------------------------------------------------------------------------------------------------------------------
# workloads
# ---------------------------------------------------------------------------------------------------------------------
def beam_bundle(wl, rank=0):
    import torj_jl_b200 as tj
    w = WORKLOADS[wl]
    pol = np.deg2rad(30.0 - 1.5 * rank)  # weak scaling: every rank its own beam
    N0 = tj.pol_tor_angles_2_vector(pol, 0.0)
    return tj.launch_peripheral_rays(np.array([2.5, 0.0, 0.4]), N0, 0.0174, 1 / 3.99, w["f"], N_rings=w["N_rings"],
                                     min_azimuthal_points=w["min_az"])


def sweep_angles():
    return [(p, t) for p in np.deg2rad(np.linspace(10.0, 40.0, 32)) for t in np.deg2rad(np.linspace(-15.0, 15.0, 32))]


def sweep_beam(b):
    import torj_jl_b200 as tj
    pol, tor = sweep_angles()[b]
    return tj.launch_peripheral_rays(np.array([2.5, 0.0, 0.4]), tj.pol_tor_angles_2_vector(pol, tor), 0.0174, 1 / 3.99, 95e9,
                                     N_rings=7, min_azimuthal_points=20)


_SWEEP = []


def sweep_bundle():
    """BASELINE.json configs[3]: all 1 049 600 rays in launch order (beam b = rays b*1025 ... b*1025+1024)."""
    if not _SWEEP:
        P, D, W = zip(*[sweep_beam(b) for b in range(1024)])
        _SWEEP.append((np.concatenate(P), np.concatenate(D), np.concatenate(W) / 1024.0))
    return _SWEEP[0]


def config5_groups(n_angles):
    """configs[4]: per T_e0 one equilibrium and one bundle of 2 launchers x 2 frequencies x n_angles beams, per-ray frequency.
    Returns [(Te0, pos, dirs, w, f_per_ray, beam_id, n_beams)]."""
    import torj_jl_b200 as tj
    out = []
    pols = np.deg2rad(30.0 + 8.0 * (np.arange(n_angles) - (n_angles - 1) / 2.0) / max(n_angles, 1))
    for te0 in (10e3, 15e3, 25e3):
        P, D, W, F, B = [], [], [], [], []
        b = 0
        for z in (0.4, -0.4):
            for f in (110e9, 170e9):
                for pol in pols:
                    N0 = tj.pol_tor_angles_2_vector(pol if z > 0 else -pol, 0.0)
                    p, d, w = tj.launch_peripheral_rays(np.array([2.5, 0.0, z]), N0, 0.0174, 1 / 3.99, f, N_rings=7, min_azimuthal_points=20)
                    P.append(p); D.append(d); W.append(w); F.append(np.full(len(w), f)); B.append(np.full(len(w), b, dtype=np.int32))
                    b += 1
        out.append((te0, np.concatenate(P), np.concatenate(D), np.concatenate(W), np.concatenate(F), np.concatenate(B), b))
    return out


def hot_arrays(te0):
    import torj_jl_b200 as tj
    arr = tj.solovev_arrays(GRID, GRID)
    arr["Te_prof"] = te0 * (1.0 - arr["psi_prof"]) ** 2 + 50.0
    return arr


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of k_trace per launch, from the committed ncu --set full capture of
    this command (profiles/ktrace_traffic.json), or None."""
    try:
        with open(os.path.join(ROOT, "profiles", "ktrace_traffic.json")) as fh:
            return float(json.load(fh)["dram_bytes_per_launch"])
    except Exception:
        return None


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self._halt = index, [], threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self._halt.wait(0.2)

    def stop(self):
        self._halt.set()
        self.join(timeout=6)
        sm = [float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(self.rows)}


def cpu_model():
    """`model name` of /proc/cpuinfo (SURVEY.md §8(d): the CPU baseline names the host it ran on)."""
    try:
        with open("/proc/cpuinfo") as fh:
            for ln in fh:
                if ln.lower().startswith("model name"):
                    return ln.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


# ---------------------------------------------------------------------------------------------------------------------
# CPU arm (oracle port; the checker doubles as the reference arm because the Julia reference cannot run here)
# ---------------------------------------------------------------------------------------------------------------------
def cpu_sample(wl, args, seconds_target):
    """(oracle plasma, pos, dirs, w, f, model): a bounded, evenly spaced sample of the workload's rays."""
    import torj_jl_b200 as tj
    from oracle import torj_oracle as O
    cores = len(os.sched_getaffinity(0))
    w = WORKLOADS[wl]
    if wl == "config5":
        te0, pos, dirs, wt, f, _, _ = config5_groups(args.c5_angles)[0]
        arr, per_ray_s = hot_arrays(te0), 12.0      # ~0.15 ms per alpha call, ~8e4 calls per ray
    else:
        arr, per_ray_s, f = tj.solovev_arrays(GRID, GRID), 0.3, w["f"]
        pos, dirs, wt = sweep_bundle() if wl == "sweep1m" else beam_bundle(wl)
    n_sample = int(max(cores, min(len(wt), round(seconds_target * cores / per_ray_s))))
    pick = np.linspace(0, len(wt) - 1, n_sample).astype(int)
    return O.OraclePlasma(*arr.values()), pos[pick], dirs[pick], wt[pick], (f[pick] if np.ndim(f) else f), w["model"], len(wt), cores


def cpu_baseline(wl, args, seconds_target=15.0, pruned_too=True):
    """Oracle port on all host cores over a bounded sample of the same workload: `value` with the reference's arithmetic
    (every harmonic integral, the reference's spline-root deposition), `value_same_work_rules` with the CUDA path's
    alpha_floor pruning and streaming deposition restated on the CPU (hardware-only comparison)."""
    from oracle import torj_oracle as O
    opl, pos, dirs, w, f, model, n_all, cores = cpu_sample(wl, args, seconds_target)
    gl = np.polynomial.legendre.leggauss(N_GL)
    psi = np.linspace(0.0, 1.0, N_PSI)
    mode = 1
    t0 = time.perf_counter()
    r = opl.trace_bundle(pos, dirs, w, f, mode, S_MAX, psi, gl, opts=O.OracleOptions.default(absorption_model=model),
                         deposition="faithful", n_threads=cores)
    dt = time.perf_counter() - t0
    out = dict(value=r["counters"]["n_acc"] / dt, unit="ray-steps/s", cores=cores, kind="port", cpu=cpu_model(),
               sample=f"{len(w)} of {n_all} rays of the same workload, evenly spaced; reference arithmetic (alpha_floor = 0, "
                      f"spline-root deposition); {dt:.1f} s", sample_rays=len(w), seconds=dt, rays_per_s=len(w) / dt,
               steps=int(r["counters"]["n_acc"]))
    if pruned_too and model == 0:
        t1 = time.perf_counter()
        r2 = opl.trace_bundle(pos, dirs, w, f, mode, S_MAX, psi, gl, opts=O.OracleOptions.default(alpha_floor=1e-14),
                              deposition="streaming", n_threads=cores)
        dt2 = time.perf_counter() - t1
        out.update(value_same_work_rules=r2["counters"]["n_acc"] / dt2,
                   same_work_rules="alpha_floor = 1e-14 harmonic pruning + inner-stage alpha skip + streaming deposition, as the "
                                   f"CUDA path; {dt2:.1f} s; absorbed fraction differs by {abs(r2['deposited_power'] - r['deposited_power']):.1e}")
    return out


def run_reference_arm(args, wl):
    """CPU arm: the reference's algorithm (oracle port; Julia is unavailable) on all host cores, bounded sample per step."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    vals, last = [], None
    for i in range(args.warmup + args.steps):
        last = cpu_baseline(wl, args, seconds_target=4.0, pruned_too=(i == args.warmup + args.steps - 1))
        if i >= args.warmup:
            vals.append(last)
    v = float(np.mean([x["value"] for x in vals]))
    ms = float(np.mean([x["seconds"] for x in vals])) * 1e3
    cb = {k: last[k] for k in ("unit", "cores", "cpu", "kind", "sample", "sample_rays") if k in last}
    cb["value"] = v
    for k in ("value_same_work_rules", "same_work_rules"):
        if k in last:
            cb[k] = last[k]
    line = {"metric": "ray-steps/s", "value": v, "unit": "ray-steps/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": WORKLOADS[wl]["scaling"],
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "impl": "reference", "config": make_config(wl, args),
            "note": "Julia reference not runnable here (no Julia); CPU oracle port, OpenMP over rays; a step is a bounded sample "
                    "of the workload (cpu_baseline.sample)",
            "cpu_baseline": cb, "rays_per_s": float(np.mean([x["rays_per_s"] for x in vals])),
            "e2e": {"value": v, "unit": "ray-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------------
# parity check (outside the timed region): the N-rank result against a host sum and against the CPU oracle
# ---------------------------------------------------------------------------------------------------------------------
def parity_check(wl, tj, pl, ctx, opt, pos_all, dirs_all, w_all, sharding, block, world, rank, device, n_pick=256):
    """(a) the all-reduced [dP_dV | deposited | sum w] equals the host sum of the per-rank vectors; (b) >= 256 rays spread
    evenly over the WHOLE bundle: step counts and final power against the oracle; (c) profiles: 4 whole beams of the sweep
    (or the 256-ray sub-bundle of a single beam) against the oracle's faithful spline-root deposition."""
    import torch.distributed as dist
    from oracle import torj_oracle as O
    from torj_jl_b200.distributed import trace_sharded
    psi = np.linspace(0.0, 1.0, N_PSI)
    f, mode = WORKLOADS[wl]["f"], WORKLOADS[wl]["mode"]
    trace = lambda p, d, w: tj.trace_bundle(pl, p, d, w, f, mode, S_MAX, psi, ctx=ctx, options=opt)
    r = trace_sharded(trace, pos_all, dirs_all, w_all, sharding=sharding, block=block, device=device)
    parts = [None] * world
    if world > 1:
        dist.all_gather_object(parts, r["local_vector"])
    else:
        parts = [r["local_vector"]]
    out = {"ranks": world}
    if rank == 0:
        host_sum = np.sum(parts, axis=0)
        got = np.concatenate([r["dP_dV"], [r["deposited_power"], r["sum_weights"]]])
        out["allreduce_vs_host_sum"] = float(np.max(np.abs(got - host_sum)) / np.max(np.abs(host_sum)))
        cores = len(os.sched_getaffinity(0))
        opl = O.OraclePlasma(*tj.solovev_arrays(GRID, GRID).values())
        gl = np.polynomial.legendre.leggauss(N_GL)
        n = len(w_all)
        pick = np.linspace(0, n - 1, n_pick).astype(int)
        ref = opl.trace_bundle(pos_all[pick], dirs_all[pick], w_all[pick], f, mode, S_MAX, psi, gl, deposition="faithful", n_threads=cores)
        good = ref["status"] == 0
        out["rays_checked"] = int(n_pick)
        out["status_equal"] = bool(np.array_equal(np.isin(r["status"][pick], (0, 3)), good))
        out["n_points_equal"] = bool(np.array_equal(r["n_points"][pick][good], ref["n_points"][good]))
        out["P_final_max_abs_dev"] = float(np.max(np.abs(r["P_final"][pick][good] - ref["P_final"][good])))
        l2 = lambda a, b: float(np.linalg.norm(a - b) / np.linalg.norm(b))
        if wl == "sweep1m":
            worst_l2, worst_dep, beams = 0.0, 0.0, []
            for b in (0, 341, 682, 1023):
                p, d, w = sweep_beam(b)
                rb = opl.trace_bundle(p, d, w, f, mode, S_MAX, psi, gl, deposition="faithful", n_threads=cores)
                gb = tj.trace_bundle(pl, p, d, w, f, mode, S_MAX, psi, ctx=ctx, options=opt)
                if (rb["status"] != 0).any() or rb["deposited_power"] < 1e-6:
                    continue
                beams.append(b)
                worst_l2 = max(worst_l2, l2(gb["dP_dV"], rb["dP_dV"]))
                worst_dep = max(worst_dep, abs(gb["deposited_power"] - rb["deposited_power"]) / rb["deposited_power"])
            out.update(beams_checked=beams, profile_l2_vs_faithful=worst_l2, absorbed_rel_dev=worst_dep)
        else:
            sub = tj.trace_bundle(pl, pos_all[pick], dirs_all[pick], w_all[pick], f, mode, S_MAX, psi, ctx=ctx, options=opt)
            out.update(profile_l2_vs_faithful=l2(sub["dP_dV"], ref["dP_dV"]),
                       absorbed_rel_dev=abs(sub["deposited_power"] - ref["deposited_power"]) / ref["deposited_power"])
        out["tolerances"] = {"allreduce": 1e-12, "P_final": 1e-11, "profile_l2": 1e-4, "absorbed_rel": 1e-6}
        out["pass"] = bool(out["allreduce_vs_host_sum"] <= 1e-12 and out["status_equal"] and out["n_points_equal"]
                           and out["P_final_max_abs_dev"] <= 1e-11 and out["profile_l2_vs_faithful"] <= 1e-4
                           and out["absorbed_rel_dev"] <= 1e-6)
        out["absorbed_fraction"] = r["deposited_power"] / r["sum_weights"]
    return out


# ---------------------------------------------------------------------------------------------------------------------
# GPU arm, one process per GPU
# ---------------------------------------------------------------------------------------------------------------------
class DeviceBundle:
    """A resident bundle (inputs in HBM before the timed region) and its step."""

    def __init__(self, L, _lib, ctx, ph, pos, dirs, w, f, mode, opt, beam_id=None, n_beams=1):
        self.L, self._lib, self.ph, self.opt = L, _lib, ph, opt
        dp = lambda a: a.ctypes.data_as(_lib.c_dp)
        self.n = len(w)
        self.keep = [np.ascontiguousarray(pos.T), np.ascontiguousarray(dirs.T), np.ascontiguousarray(w)]
        per_ray = int(np.ndim(f) > 0)
        fr = np.ascontiguousarray(np.atleast_1d(f), dtype=np.float64)
        md = np.ascontiguousarray(np.broadcast_to(np.atleast_1d(mode), fr.shape), dtype=np.int32)
        self.bh = _lib.c_vp()
        _lib.check(L.torj_bundle_create(ctx, self.n, dp(self.keep[0]), dp(self.keep[1]), dp(self.keep[2]), dp(fr),
                                        md.ctypes.data_as(_lib.c_ip), per_ray, C.byref(self.bh)))
        if beam_id is not None:
            bid = np.ascontiguousarray(beam_id, dtype=np.int32)
            _lib.check(L.torj_bundle_set_beams(self.bh, int(n_beams), bid.ctypes.data_as(_lib.c_ip)))
        self.n_beams = int(n_beams) if beam_id is not None else 1
        self.psi = np.ascontiguousarray(np.linspace(0.0, 1.0, N_PSI))

    def step(self, opt=None):
        o = opt or self.opt
        self._lib.check(self.L.torj_bundle_trace(self.bh, self.ph, C.byref(o), S_MAX, N_PSI, self.psi.ctypes.data_as(self._lib.c_dp)))

    def profile_tensor(self, torch, local):
        class _DevBuf:
            __cuda_array_interface__ = {"shape": (self.n_beams * (N_PSI + 2),), "typestr": "<f8", "version": 2,
                                        "data": (int(self.L.torj_bundle_device_profile(self.bh)), False)}
        return torch.as_tensor(_DevBuf(), device=torch.device("cuda", local))

    def counters(self):
        cnt = self._lib.TorjCounters()
        dep = np.zeros(self.n_beams)
        st = np.zeros(self.n, dtype=np.int32)
        self._lib.check(self.L.torj_bundle_results(self.bh, None, dep.ctypes.data_as(self._lib.c_dp), None, None, None,
                                                   st.ctypes.data_as(self._lib.c_ip), C.byref(cnt)))
        return cnt.as_dict(), dep, st

    def results(self):
        """Every array torj_bundle_results hands its caller after the last trace, and the counters."""
        dp, ip = (lambda a: a.ctypes.data_as(self._lib.c_dp)), (lambda a: a.ctypes.data_as(self._lib.c_ip))
        r = dict(dP_dV=np.zeros((self.n_beams, N_PSI)), deposited_power=np.zeros(self.n_beams), P_final=np.zeros(self.n),
                 P_deposited_ray=np.zeros(self.n), n_points=np.zeros(self.n, dtype=np.int32), status=np.zeros(self.n, dtype=np.int32))
        cnt = self._lib.TorjCounters()
        self._lib.check(self.L.torj_bundle_results(self.bh, dp(r["dP_dV"]), dp(r["deposited_power"]), dp(r["P_final"]),
                                                   dp(r["P_deposited_ray"]), ip(r["n_points"]), ip(r["status"]), C.byref(cnt)))
        r["counters"] = np.array(list(cnt.as_dict().values()))
        return r

    def close(self):
        self.L.torj_bundle_destroy(self.bh)


PER_RAY = ("P_final", "P_deposited_ray", "n_points", "status")


def dump_outputs(out_dir, bundles, rank, world, budget=64_000_000):
    """--dump-outputs: the results of the last timed step as float64 .npy files, rays of several bundles concatenated,
    profile rows stacked and counters summed; under several ranks each rank writes its own, prefixed rank<r>_. Per-ray
    arrays that would take the file set over `budget` bytes are cut to a fixed seeded sample of rays, whose indices go to
    ray_index.npy."""
    rs = [b.results() for b in bundles]
    out = {k: np.concatenate([r[k] for r in rs]).astype(np.float64) for k in rs[0] if k != "counters"}
    out["counters"] = np.sum([r["counters"] for r in rs], axis=0).astype(np.float64)
    n = len(out["P_final"])
    fixed = sum(v.nbytes for k, v in out.items() if k not in PER_RAY)
    if n * 8 * len(PER_RAY) > budget // world - fixed:
        keep = (budget // world - fixed) // (8 * (len(PER_RAY) + 1))
        idx = np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
        out.update({k: out[k][idx] for k in PER_RAY}, ray_index=idx.astype(np.float64))
    os.makedirs(out_dir, exist_ok=True)
    prefix = f"rank{rank}_" if world > 1 else ""
    for k, v in out.items():
        np.save(os.path.join(out_dir, f"{prefix}{k}.npy"), v)


def run_gpu_arm(args, wl):
    import torch
    import torch.distributed as dist
    import torj_jl_b200 as tj
    from torj_jl_b200 import _lib
    from torj_jl_b200.distributed import shard_indices

    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    W = WORKLOADS[wl]
    model = W["model"]
    L = tj.lib()
    tstream = torch.cuda.Stream()  # the library launches on this torch stream so torch events bracket its kernels
    torch.cuda.set_stream(tstream)
    ctx = _lib.context(local, tstream.cuda_stream)
    tj.abs_Al_init(N_GL, ctx)
    opt = _lib.default_options(schedule=args.schedule, absorption_model=model, lanes_per_ray=args.lanes_per_ray)
    opt_exact = _lib.default_options(schedule=args.schedule, absorption_model=model, lanes_per_ray=args.lanes_per_ray, alpha_floor=0.0)

    # ---- this rank's resident bundle(s)
    pos_all = dirs_all = w_all = None
    sharding, block = "contiguous", 1
    bundles, plasmas = [], []
    if wl == "config5":
        for te0, pos, dirs, w, f, bid, nb in config5_groups(args.c5_angles):
            pl = tj.Plasma(*hot_arrays(te0).values(), build="device")
            idx = shard_indices(len(w), rank, world, "block_cyclic", C5_BLOCK)
            plasmas.append(pl)
            bundles.append(DeviceBundle(L, _lib, ctx, pl.handle(ctx), pos[idx], dirs[idx], w[idx], f[idx], 1, opt, bid[idx], nb))
    else:
        pl = tj.Plasma(*tj.solovev_arrays(GRID, GRID).values())
        plasmas.append(pl)
        if wl == "sweep1m":
            pos_all, dirs_all, w_all = sweep_bundle()
            sharding, block = "block_cyclic", 1025
            idx = shard_indices(len(w_all), rank, world, sharding, block)
            pos, dirs, w = pos_all[idx], dirs_all[idx], w_all[idx]
        else:
            pos, dirs, w = beam_bundle(wl, rank)
            pos_all, dirs_all, w_all = beam_bundle(wl, 0)  # the parity check shards rank 0's beam over all ranks
        bundles.append(DeviceBundle(L, _lib, ctx, pl.handle(ctx), pos, dirs, w, W["f"], W["mode"], opt))
    n = sum(b.n for b in bundles)
    prof_t = [None] * len(bundles)

    def device_step(o=None):
        for i, b in enumerate(bundles):
            b.step(o)
            if world > 1:
                if prof_t[i] is None:
                    prof_t[i] = b.profile_tensor(torch, local)  # the library's device buffer as a torch tensor (no copy)
                dist.all_reduce(prof_t[i])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(nsteps, o=None):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        barrier()
        ev[0].record()
        for _ in range(nsteps):
            device_step(o)
        ev[1].record()
        barrier()
        return ev[0].elapsed_time(ev[1])

    for _ in range(args.warmup):
        device_step()
    barrier()
    launches0 = L.torj_ctx_launch_count(ctx)
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    ms_total = timed(args.steps)
    clocks = sampler.stop() if sampler else None
    launches = L.torj_ctx_launch_count(ctx) - launches0
    c = {}
    for b in bundles:
        cb, _, _ = b.counters()
        for k, v in cb.items():
            c[k] = c.get(k, 0) + v
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, bundles, rank, world)  # before the alpha_floor = 0 pass below traces the bundles again
    kms = C.c_double()
    _lib.check(L.torj_ctx_last_trace_ms(ctx, C.byref(kms)))  # the last trace kernel alone, CUDA events on its own stream

    # ---- the same bundle with alpha_floor = 0: every harmonic integral / every warm quadrature evaluated (reference arithmetic)
    n_exact = 0 if args.no_exact else max(1, min(args.steps, 2 if wl != "config5" else 1))
    exact_ms = None
    if n_exact:
        device_step(opt_exact)
        exact_ms = timed(n_exact, opt_exact) / n_exact
        device_step()  # leave the bundle as the default options traced it

    # ---- end to end through the reference-facing call with HOST buffers (H2D of the bundle, D2H of the results)
    e2e = None
    if wl != "config5":
        psi = np.linspace(0.0, 1.0, N_PSI)

        def e2e_step():
            r = tj.trace_bundle(plasmas[0], pos, dirs, w, W["f"], W["mode"], S_MAX, psi, ctx=ctx, options=opt)
            if world > 1:
                t = torch.from_numpy(np.concatenate([r["dP_dV"], [r["deposited_power"], w.sum()]])).cuda()
                dist.all_reduce(t)
                t.cpu()
            return r
        e2e_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            e2e_step()
        barrier()
        e2e_s = (time.perf_counter() - t0) / args.steps
        e2e = dict(ms=e2e_s * 1e3, h2d=8 * (3 * n + 3 * n + n + 1 + N_PSI) + 4, d2h=8 * (N_PSI + 2 + 2 * n) + 4 * 2 * n + 48)
    else:
        def e2e_step():
            for (te0, p5, d5, w5, f5, b5, nb), plq in zip(groups5, plasmas):
                tj.trace_bundle(plq, p5, d5, w5, f5, 1, S_MAX, np.linspace(0.0, 1.0, N_PSI), ctx=ctx, options=opt, beam_id=b5, n_beams=nb)
        groups5 = [(te0, p5[i5], d5[i5], w5[i5], f5[i5], b5[i5], nb) for (te0, p5, d5, w5, f5, b5, nb) in config5_groups(args.c5_angles)
                   for i5 in [shard_indices(len(w5), rank, world, "block_cyclic", C5_BLOCK)]]
        barrier()
        t0 = time.perf_counter()
        e2e_step()
        barrier()
        e2e = dict(ms=(time.perf_counter() - t0) * 1e3, h2d=8 * 8 * n + 4 * n, d2h=8 * 2 * n + 8 * n)

    # ---- parity (outside every timed region)
    par = None
    if not args.no_parity and wl != "config5":
        par = parity_check(wl, tj, plasmas[0], ctx, opt, pos_all, dirs_all, w_all, sharding, block, world, rank,
                           torch.device("cuda", local) if world > 1 else None)
    elif not args.no_parity:
        par = parity_check_config5(tj, plasmas, ctx, opt, args, rank)

    # ---- max over ranks
    t_ms = torch.tensor([ms_total, e2e["ms"], exact_ms or 0.0], dtype=torch.float64, device="cuda")
    tot = torch.tensor([c["n_acc"], n, algorithmic_flops(c, model)], dtype=torch.float64, device="cuda")
    rays_ok = torch.tensor([c["n_rays_ok"]], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot)
        dist.all_reduce(rays_ok)
    ms_total, e2e_ms, exact_ms_max = t_ms.tolist()
    steps_all, rays_all, flops_all = tot.tolist()
    ms_per_step = ms_total / args.steps

    if rank == 0:
        tf, tms = C.c_double(), C.c_double()
        _lib.check(L.torj_fp64_peak(ctx, 20000, C.byref(tf), C.byref(tms)))
        # roofline of the dominant kernel (k_trace) on this rank: algorithmic FP64 flops / step time; k_ray_init and
        # k_finalize are < 1 % of the step (profiles/), so the step time stands for the kernel
        achieved = algorithmic_flops(c, model) / (ms_per_step * 1e-3) / 1e12
        kname = "k_trace<Tsit5" + (", warm" if model else "") + ">"
        roof = {"bound": "fp64", "achieved": achieved, "peak": tf.value, "unit": "TFLOP/s", "frac": achieved / tf.value,
                "traffic": ncu_traffic() if wl == "beam64k" else None, "kernel": kname, "kernel_ms_last_launch": kms.value,
                "peak_source": "DFMA-chain microbenchmark torj_fp64_peak measured in this run (MEASURED_PEAKS.json has no FP64 entry)",
                "algorithmic_flops_per_launch": algorithmic_flops(c, model), "counters": c}
        cfg = make_config(wl, args)
        line = {"metric": "ray-steps/s", "value": steps_all / (ms_per_step * 1e-3), "unit": "ray-steps/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
                "scaling": W["scaling"], "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": cfg,
                "sharding": {"n_rays_this_gpu": n, "kind": "one beam per rank" if W["scaling"] == "weak" else
                             (f"{C5_BLOCK}-ray blocks dealt round-robin: every rank traces 1/N of every beam" if wl == "config5" else
                              "beams dealt round-robin (block-cyclic, 1025 rays)"),
                             "schedule": args.schedule, "lanes_per_ray": args.lanes_per_ray},
                "rays_per_s": rays_all / (ms_per_step * 1e-3), "rays_total": int(rays_all), "rays_ok": int(rays_ok.item()),
                "e2e": {"value": steps_all / (e2e_ms * 1e-3), "unit": "ray-steps/s", "h2d_bytes_per_step": e2e["h2d"],
                        "d2h_bytes_per_step": e2e["d2h"], "ms_per_step": e2e_ms, "rays_per_s": rays_all / (e2e_ms * 1e-3)},
                "gpu_launches": int(launches), "clocks": clocks, "roofline": roof}
        if n_exact:
            line["exact_ms_per_step"] = exact_ms_max
            line["exact_value"] = steps_all / (exact_ms_max * 1e-3)
            line["exact_note"] = ("same bundle with torj_options.alpha_floor = 0: every harmonic integral / warm quadrature evaluated as "
                                  "the reference does (the default prunes those below 1e-14 1/m); compare with cpu_baseline.value")
        if par is not None:
            line["parity_check"] = par
        if not args.no_cpu_baseline:
            line["cpu_baseline"] = {k: v for k, v in cpu_baseline(wl, args).items() if k not in ("seconds", "steps")}
        if wl == "beam64k" and world == 1 and not args.no_anchor:
            line["strong_scaling_n1"] = sweep_anchor(L, _lib, tj, ctx, plasmas[0], opt, torch)
        print(json.dumps(line), flush=True)
    for b in bundles:
        b.close()
    bad = par is not None and rank == 0 and not par.get("pass", True)
    if world > 1:
        flag = torch.tensor([1.0 if bad else 0.0], device="cuda")
        dist.all_reduce(flag)
        bad = flag.item() > 0
        dist.barrier()
        dist.destroy_process_group()
    if bad:
        print("bench.py: parity check FAILED", file=sys.stderr, flush=True)
        sys.exit(3)


def sweep_anchor(L, _lib, tj, ctx, pl, opt, torch):
    """N = 1 point of the strong-scaling curve the N > 1 runs measure (configs[3], 1 049 600 rays): 1 warm-up + 2 steps."""
    pos, dirs, w = sweep_bundle()
    b = DeviceBundle(L, _lib, ctx, pl.handle(ctx), pos, dirs, w, 95e9, 1, opt)
    try:
        b.step()
        torch.cuda.synchronize()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        ev[0].record()
        b.step(); b.step()
        ev[1].record()
        torch.cuda.synchronize()
        ms = ev[0].elapsed_time(ev[1]) / 2.0
        c, _, _ = b.counters()
        return {"workload": WORKLOADS["sweep1m"]["name"], "n_rays": b.n, "ms_per_step": ms, "value": c["n_acc"] / (ms * 1e-3),
                "rays_per_s": b.n / (ms * 1e-3), "steps": 2, "warmup": 1}
    finally:
        b.close()


def parity_check_config5(tj, plasmas, ctx, opt, args, rank):
    """Warm model: 3 rays per (T_e0, launcher, frequency) against the oracle's make_ray with absorption_model = 1 (the
    oracle needs ~10 s per ray), absorbed fraction of each ray rel 1e-6."""
    if rank != 0:
        return {}
    from oracle import torj_oracle as O
    cores = len(os.sched_getaffinity(0))
    gl = np.polynomial.legendre.leggauss(N_GL)
    psi = np.linspace(0.0, 1.0, N_PSI)
    worst, n_chk, npts_ok = 0.0, 0, True
    for (te0, pos, dirs, w, f, bid, nb), pl in zip(config5_groups(1), plasmas):
        pick = np.concatenate([b * 1025 + np.array([0, 500, 1024]) for b in range(nb)])
        opl = O.OraclePlasma(*hot_arrays(te0).values())
        ref = opl.trace_bundle(pos[pick], dirs[pick], np.ones(len(pick)), f[pick], 1, S_MAX, psi, gl,
                               opts=O.OracleOptions.default(absorption_model=1), deposition="streaming", n_threads=cores)
        got = tj.trace_bundle(pl, pos[pick], dirs[pick], np.ones(len(pick)), f[pick], 1, S_MAX, psi, ctx=ctx, options=opt)
        good = ref["status"] == 0
        npts_ok = npts_ok and bool(np.array_equal(got["n_points"][good], ref["n_points"][good]))
        absorbed_ref, absorbed = 1.0 - ref["P_final"][good], 1.0 - got["P_final"][good]
        worst = max(worst, float(np.max(np.abs(absorbed - absorbed_ref) / np.maximum(absorbed_ref, 1e-3))))
        n_chk += int(good.sum())
    return {"rays_checked": n_chk, "n_points_equal": npts_ok, "absorbed_rel_dev": worst, "tolerances": {"absorbed_rel": 1e-6},
            "pass": bool(npts_ok and worst <= 1e-6)}


# ---------------------------------------------------------------------------------------------------------------------
# ONE process, N devices: what a Julia session's make_beam binds (torj_multi_trace)
# ---------------------------------------------------------------------------------------------------------------------
def run_multi_arm(args, wl):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    import torj_jl_b200 as tj
    from torj_jl_b200 import _lib
    W = WORKLOADS[wl]
    mg = tj.MultiGPU(args.gpus)
    mg.abs_Al_init(N_GL)
    pl = tj.Plasma(*tj.solovev_arrays(GRID, GRID).values(), build="device")
    pos, dirs, w = sweep_bundle() if wl == "sweep1m" else beam_bundle(wl)
    # column-major (n, 3), the layout of a Julia Matrix[n, 3]: the library's component-major [3][n] without a copy
    pos, dirs = np.asfortranarray(pos), np.asfortranarray(dirs)
    mg.configure(sharding="block_cyclic" if wl == "sweep1m" else "contiguous", block_rays=1025, deterministic=args.deterministic)
    psi = np.linspace(0.0, 1.0, N_PSI)
    opt = _lib.default_options(schedule=args.schedule)
    r = None
    for _ in range(max(args.warmup, 1)):
        r = mg.trace_bundle(pl, pos, dirs, w, W["f"], W["mode"], S_MAX, psi, options=opt)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        r = mg.trace_bundle(pl, pos, dirs, w, W["f"], W["mode"], S_MAX, psi, options=opt)
    ms = (time.perf_counter() - t0) / args.steps * 1e3
    n = len(w)
    v = r["counters"]["n_acc"] / (ms * 1e-3)
    line = {"metric": "ray-steps/s", "value": v, "unit": "ray-steps/s", "n_gpus": mg.n_devices, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "impl": "multi", "config": make_config(wl, args),
            "timing": "host wall clock around the blocking torj_multi_trace call (host buffers in Julia's column-major layout, results out): an end-to-end number",
            "collective": "ncclAllReduce on the devices' profile buffers" if mg.used_nccl else "host sum in device order",
            "rays_per_s": n / (ms * 1e-3), "absorbed_fraction": r["deposited_power"],
            "e2e": {"value": v, "unit": "ray-steps/s", "h2d_bytes_per_step": 8 * 7 * n, "d2h_bytes_per_step": 8 * (N_PSI + 2 + 2 * n) + 8 * n,
                    "ms_per_step": ms}}
    print(json.dumps(line), flush=True)
    mg.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "multi"])
    ap.add_argument("--workload", default=None, choices=sorted(WORKLOADS),
                    help="default: beam64k at N = 1 (configs[2]), sweep1m at N > 1 (configs[3], strong scaling)")
    ap.add_argument("--small", action="store_true", help="alias of --workload small (configs[1], 1 025 rays)")
    ap.add_argument("--c5-angles", type=int, default=2, help="config5: steering angles per (launcher, frequency); 85 gives 1 045 500 rays")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-exact", action="store_true")
    ap.add_argument("--no-anchor", action="store_true")
    ap.add_argument("--deterministic", action="store_true", help="--impl multi: host sum in device order instead of NCCL")
    ap.add_argument("--schedule", type=int, default=0, choices=[0, 1, 2],
                    help="torj_options.schedule: 0 automatic (default), 1 whole rays per lane, 2 segment hand-off")
    ap.add_argument("--lanes-per-ray", type=int, default=0, choices=[0, 1, 32])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the results of the last timed step to DIR/<name>.npy (float64; default --impl only)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the results of the CUDA path of the default --impl")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    wl = args.workload or ("small" if args.small else ("sweep1m" if max(world, args.gpus) > 1 else "beam64k"))
    if args.impl == "reference":
        return run_reference_arm(args, wl)
    if args.impl == "multi":
        return run_multi_arm(args, wl)
    return run_gpu_arm(args, wl)


if __name__ == "__main__":
    main()
