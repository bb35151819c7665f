"""Exact deposition sums on the GPU (torj_ctx_set_exact_sum / torj_multi_set_exact_sum, trace calls with exact_sum=True).

Profiles and deposited powers are compared as bits. In exact mode they must not depend on the run, the schedule, the ray
order, the plasma-set grouping or the device count (at a fixed lanes_per_ray); per-ray results must equal the float
mode's bit for bit, since only the summation changes; and the deposited power must equal the Python model of the format
(tests/test_exact_sum_format.py) applied to the per-ray results."""
import ctypes as C
from fractions import Fraction

import numpy as np
import pytest

import torj_jl_b200 as tj
from torj_jl_b200 import _lib

pytestmark = pytest.mark.gpu

GRID, N_PSI, S_MAX = 257, 1000, 1.0  # the bench workload (bench.py)
PSI = np.linspace(0.0, 1.0, N_PSI)


@pytest.fixture(scope="module", autouse=True)
def _abs_al_init():
    tj.abs_Al_init(24)


@pytest.fixture(scope="module")
def plasma(arrays_full):
    return tj.Plasma(*arrays_full.values())


@pytest.fixture(scope="module")
def plasma_dev(arrays_full):
    """built like the per-device copies of MultiGPU (torj_plasma_create_from_data): the same tables bit for bit"""
    return tj.Plasma(*arrays_full.values(), build="device")


def bits(a):
    return np.ascontiguousarray(np.atleast_1d(np.asarray(a, dtype=np.float64))).view(np.uint64)


def same_bits(a, b):
    return np.array_equal(bits(a), bits(b))


def bench_bundle():
    N0 = tj.pol_tor_angles_2_vector(np.deg2rad(30.0), 0.0)
    return tj.launch_peripheral_rays(np.array([2.5, 0.0, 0.4]), N0, 0.0174, 1 / 3.99, 95e9, N_rings=66, min_azimuthal_points=14)


def multi_beam_bundle(n_beams):
    """n_beams beams of 1 025 rays at different steering angles: past the resident lanes at one lane per ray for n >= 37"""
    P, D, W, B = [], [], [], []
    for b, pol in enumerate(np.linspace(15.0, 40.0, n_beams)):
        p, d, w = tj.launch_peripheral_rays(np.array([2.5, 0.0, 0.4]), tj.pol_tor_angles_2_vector(np.deg2rad(pol), 0.02 * b),
                                            0.0174, 1 / 3.99, 95e9, N_rings=7, min_azimuthal_points=20)
        P.append(p); D.append(d); W.append(w); B.append(np.full(len(w), b, dtype=np.int32))
    return np.concatenate(P), np.concatenate(D), np.concatenate(W), np.concatenate(B)


def quantize(v):
    return round(Fraction(float(v)) * 2 ** 160)


def exact_model(vals):
    """The correctly rounded exact sum of bookings rounded to 2^-160 (torj_exactsum.cuh)"""
    return float(Fraction(sum(quantize(v) for v in vals), 2 ** 160))


def fatal(st):
    return (st != 0) & (st != 3) & (st != 6)


def test_run_to_run_bench_bundle(plasma):
    pos, dirs, w = bench_bundle()
    assert len(w) == 65543
    runs = {}
    for exact in (True, False):
        runs[exact] = [tj.trace_bundle(plasma, pos, dirs, w, 95e9, 1, S_MAX, PSI, exact_sum=exact) for _ in range(3)]
    ex = runs[True]
    for r in ex[1:]:
        assert same_bits(r["dP_dV"], ex[0]["dP_dV"]) and same_bits(r["deposited_power"], ex[0]["deposited_power"])
    fl = runs[False]
    differ = sum(not (same_bits(r["dP_dV"], fl[0]["dP_dV"]) and same_bits(r["deposited_power"], fl[0]["deposited_power"]))
                 for r in fl[1:])
    print(f"\nfloat mode: {differ} of 2 repeats differed from the first run in dP_dV / deposited_power bits")
    # end-to-end format check: deposited power = the model over fl(w_i P_deposited_ray_i) of the rays with a result
    r = ex[0]
    ok = ~fatal(r["status"])
    assert r["deposited_power"] == exact_model(w[ok] * r["P_deposited_ray"][ok])
    # against the float mode: the same per-ray results, profiles to the order of summation
    f = fl[0]
    for k in ("status", "n_points", "P_final", "P_deposited_ray"):
        assert np.array_equal(np.asarray(r[k]).view(np.uint8), np.asarray(f[k]).view(np.uint8)), k
    assert r["counters"] == f["counters"]
    scale = np.abs(f["dP_dV"]).max()
    assert np.abs(r["dP_dV"] - f["dP_dV"]).max() <= 1e-13 * scale
    assert abs(r["deposited_power"] - f["deposited_power"]) <= 1e-13 * abs(f["deposited_power"])


@pytest.fixture(scope="module")
def beams40():
    return multi_beam_bundle(40)


def test_schedules_and_ray_order(plasma, beams40):
    pos, dirs, w, bid = beams40
    assert len(w) > 148 * 2 * 128  # more rays than resident lanes at one lane per ray
    res = {}
    for sch in (1, 2, 3):
        opt = _lib.default_options(lanes_per_ray=1, schedule=sch)
        res[sch] = tj.trace_bundle(plasma, pos, dirs, w, 95e9, 1, S_MAX, PSI, options=opt, beam_id=bid, n_beams=40,
                                   exact_sum=True)
    for sch in (2, 3):
        assert same_bits(res[sch]["dP_dV"], res[1]["dP_dV"]), sch
        assert same_bits(res[sch]["deposited_power"], res[1]["deposited_power"]), sch
    perm = np.random.default_rng(5).permutation(len(w))
    opt = _lib.default_options(lanes_per_ray=1)
    rp = tj.trace_bundle(plasma, pos[perm], dirs[perm], w[perm], 95e9, 1, S_MAX, PSI, options=opt, beam_id=bid[perm],
                         n_beams=40, exact_sum=True)
    assert same_bits(rp["dP_dV"], res[1]["dP_dV"]) and same_bits(rp["deposited_power"], res[1]["deposited_power"])
    assert np.array_equal(rp["P_deposited_ray"], res[1]["P_deposited_ray"][perm])
    # each row's deposited power is the model over its own rays
    ok = ~fatal(res[1]["status"])
    for b in (0, 17, 39):
        sel = ok & (bid == b)
        assert res[1]["deposited_power"][b] == exact_model(w[sel] * res[1]["P_deposited_ray"][sel])


def test_float_mode_per_ray_outputs_and_window_are_unchanged(plasma, beams40):
    pos, dirs, w, bid = beams40
    opt = _lib.default_options(lanes_per_ray=1)
    r = {e: tj.trace_bundle(plasma, pos, dirs, w, 95e9, 1, S_MAX, PSI, options=opt, beam_id=bid, n_beams=40,
                            trajectories=(1000, 40), exact_sum=e) for e in (True, False)}
    for k in ("status", "n_points", "P_final", "P_deposited_ray", "traj_s", "traj_xyz", "traj_P", "traj_dP_ds",
              "traj_dP_dV_ray"):
        assert np.array_equal(np.asarray(r[True][k]).view(np.uint8), np.asarray(r[False][k]).view(np.uint8)), k
    assert r[True]["counters"] == r[False]["counters"]
    a, b = r[True]["dP_dV"], r[False]["dP_dV"]
    assert np.abs(a - b).max() <= 1e-13 * np.abs(b).max()
    assert np.abs(r[True]["deposited_power"] - r[False]["deposited_power"]).max() <= 1e-13 * np.abs(r[False]["deposited_power"]).max()


def test_plasma_set_rows_equal_separate_calls():
    pls = [tj.Plasma(*tj.solovev_arrays(129, 129, **kw).values()) for kw in ({}, dict(Te0=6e3), dict(B0=2.1))]
    pos, dirs, w, bid = multi_beam_bundle(4)
    bp = np.array([2, 0, 1, 2], dtype=np.int32)
    opt = _lib.default_options(lanes_per_ray=1)
    s = tj.trace_bundle(pls, pos, dirs, w, 95e9, 1, S_MAX, PSI, options=opt, beam_id=bid, n_beams=4, beam_plasma=bp,
                        exact_sum=True)
    for b in range(4):
        sel = bid == b
        one = tj.trace_bundle(pls[bp[b]], pos[sel], dirs[sel], w[sel], 95e9, 1, S_MAX, PSI, options=opt, exact_sum=True)
        assert same_bits(s["dP_dV"][b], one["dP_dV"]), b
        assert same_bits(s["deposited_power"][b], one["deposited_power"]), b


def test_warm_model_run_to_run():
    pl = tj.Plasma(*tj.solovev_arrays(129, 129, Te0=10e3).values())
    N0 = tj.pol_tor_angles_2_vector(np.deg2rad(30.0), 0.0)
    pos, dirs, w = tj.launch_peripheral_rays(np.array([2.5, 0.0, 0.4]), N0, 0.0174, 1 / 3.99, 95e9)
    opt = _lib.default_options(absorption_model=1, lanes_per_ray=32)
    r = [tj.trace_bundle(pl, pos, dirs, w, 95e9, 1, 0.6, PSI, options=opt, exact_sum=True) for _ in range(3)]
    assert r[0]["deposited_power"] > 0
    for q in r[1:]:
        assert same_bits(q["dP_dV"], r[0]["dP_dV"]) and same_bits(q["deposited_power"], r[0]["deposited_power"])
    ok = ~fatal(r[0]["status"])
    assert r[0]["deposited_power"] == exact_model(w[ok] * r[0]["P_deposited_ray"][ok])


def test_multi_device_equals_one_device(plasma_dev, beams40):
    plasma = plasma_dev
    pos, dirs, w, bid = beams40
    opt = _lib.default_options(lanes_per_ray=1)
    one = tj.trace_bundle(plasma, pos, dirs, w, 95e9, 1, S_MAX, PSI, options=opt, beam_id=bid, n_beams=40, exact_sum=True)
    mg = tj.MultiGPU()
    try:
        mg.abs_Al_init(24)
        print(f"\nMultiGPU over {mg.n_devices} visible device(s)")
        for sharding, block in (("contiguous", 1), ("block_cyclic", 1025)):
            for det in (False, True):
                mg.configure(sharding, block, det)
                r = mg.trace_bundle(plasma, pos, dirs, w, 95e9, 1, S_MAX, PSI, options=opt, beam_id=bid, n_beams=40,
                                    exact_sum=True)
                assert same_bits(r["dP_dV"], one["dP_dV"]), (sharding, det, mg.used_nccl)
                assert same_bits(r["deposited_power"], one["deposited_power"]), (sharding, det, mg.used_nccl)
                assert np.array_equal(r["P_deposited_ray"], one["P_deposited_ray"])
                if mg.n_devices > 1 and not det:
                    print(f"{sharding}: NCCL used = {mg.used_nccl}")
        assert set(mg.config) == {"sharding", "block_rays", "deterministic"}
    finally:
        mg.close()


def test_refusals_leave_the_earlier_results(plasma):
    N0 = tj.pol_tor_angles_2_vector(np.deg2rad(30.0), 0.0)
    pos, dirs, w = tj.launch_peripheral_rays(np.array([2.5, 0.0, 0.4]), N0, 0.0174, 1 / 3.99, 95e9)
    L, ctx = tj.lib(), _lib.context()
    ref = tj.trace_bundle(plasma, pos, dirs, w, 95e9, 1, S_MAX, PSI, exact_sum=True)
    for bad in (2, -1):
        assert L.torj_ctx_set_exact_sum(ctx, bad) != 0
        assert b"on must be 0" in L.torj_last_error()
        r = tj.trace_bundle(plasma, pos, dirs, w, 95e9, 1, S_MAX, PSI, exact_sum=True)
        assert same_bits(r["dP_dV"], ref["dP_dV"]) and same_bits(r["deposited_power"], ref["deposited_power"])
    # weights beyond the accepted range are refused before anything runs, then a valid call gives the same bits
    big = w.copy()
    big[3] = 2.0 ** 41
    with pytest.raises(_lib.TorjError, match="2\\^40"):
        tj.trace_bundle(plasma, pos, dirs, big, 95e9, 1, S_MAX, PSI, exact_sum=True)
    r = tj.trace_bundle(plasma, pos, dirs, w, 95e9, 1, S_MAX, PSI, exact_sum=True)
    assert same_bits(r["dP_dV"], ref["dP_dV"]) and same_bits(r["deposited_power"], ref["deposited_power"])
    # the float mode takes such weights as before
    tj.trace_bundle(plasma, pos, dirs, big, 95e9, 1, S_MAX, PSI)
    mg = tj.MultiGPU()
    try:
        mg.abs_Al_init(24)
        m0 = mg.trace_bundle(plasma, pos, dirs, w, 95e9, 1, S_MAX, PSI, exact_sum=True)
        assert L.torj_multi_set_exact_sum(mg.h, 2) != 0
        assert b"on must be 0" in L.torj_last_error()
        m1 = mg.trace_bundle(plasma, pos, dirs, w, 95e9, 1, S_MAX, PSI, exact_sum=True)
        assert same_bits(m1["dP_dV"], m0["dP_dV"]) and same_bits(m1["deposited_power"], m0["deposited_power"])
    finally:
        mg.close()
