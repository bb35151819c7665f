"""Segment hand-off (torj_options.schedule 0 / 2 / 3) against whole rays per lane (schedule 1).

The hand-off only decides which lane runs which segment of a ray. So with lanes_per_ray pinned, every per-ray output must
equal that of whole-ray tracing bit for bit: status, n_points, P_final, P_deposited_ray, the final state, the trajectory
window, and the step and ray counters; the profiles agree to the order of their atomic sums. A segment run twice, skipped
or lost would show here. The runs force the hand-off where the protocol's races are most likely: small bundles with up to
16 000 segments (a hand-in every step or two), life-ordered rounds over rays of very different lives, the warm model and a
plasma set. Every run is also checked on its own: counted rays, each beam's power against its rays, and no jump of a
trajectory beyond dtmax."""
import ctypes as C

import numpy as np
import pytest

import torj_jl_b200 as tj
from oracle import torj_oracle as O
from torj_jl_b200 import _lib

pytestmark = pytest.mark.gpu

PSI = np.linspace(0.0, 1.0, 200)


@pytest.fixture(scope="module", autouse=True)
def _abs_al_init():
    tj.abs_Al_init(24)


@pytest.fixture(scope="module")
def gpu_full(arrays_full):
    return tj.Plasma(*arrays_full.values())


def dp(a):
    return a.ctypes.data_as(_lib.c_dp)


def ip(a):
    return a.ctypes.data_as(_lib.c_ip)


def fatal(st):
    """status codes that end a ray without a result (include/torj_cuda.h): all but OK, LEFT_GRID and TRAJ_TRUNCATED"""
    return (st != 0) & (st != 3) & (st != 6)


def max_points(opt, s_max):
    return 2 + int(opt.n_segments * (np.ceil(s_max / opt.n_segments / opt.dtmax) + 8))


def run(plasmas, pos, dirs, w, f, mode, s_max, opt, window, beam_id=None, n_beams=1, beam_plasma=None):
    """One resident bundle through torj_bundle_trace (a Plasma) or torj_bundle_trace_plasmas (a list): results, counters,
    final states and the trajectories of the rays window = (first, count); checked on its own before it is returned."""
    L = tj.lib()
    ctx = _lib.context()
    n = len(w)
    posT = np.ascontiguousarray(np.asarray(pos, dtype=np.float64).T)
    dirT = np.ascontiguousarray(np.asarray(dirs, dtype=np.float64).T)
    w = np.ascontiguousarray(w, dtype=np.float64)
    per_ray = int(np.ndim(f) > 0)
    fr = np.ascontiguousarray(np.atleast_1d(f), dtype=np.float64)
    md = np.ascontiguousarray(np.broadcast_to(np.atleast_1d(mode), fr.shape), dtype=np.int32)
    first, count = window
    mp = max_points(opt, s_max)
    bh = _lib.c_vp()
    _lib.check(L.torj_bundle_create(ctx, n, dp(posT), dp(dirT), dp(w), dp(fr), ip(md), per_ray, C.byref(bh)))
    try:
        _lib.check(L.torj_bundle_set_window(bh, first, count, mp))
        if beam_id is not None:
            _lib.check(L.torj_bundle_set_beams(bh, n_beams, ip(np.ascontiguousarray(beam_id, dtype=np.int32))))
        if isinstance(plasmas, tj.Plasma):
            _lib.check(L.torj_bundle_trace(bh, plasmas.handle(ctx), C.byref(opt), s_max, len(PSI), dp(PSI)))
        else:
            hs = (_lib.c_vp * len(plasmas))(*[p.handle(ctx).value for p in plasmas])
            bp = np.ascontiguousarray(beam_plasma, dtype=np.int32)
            _lib.check(L.torj_bundle_trace_plasmas(bh, len(plasmas), hs, ip(bp), C.byref(opt), s_max, len(PSI), dp(PSI)))
        prof = np.zeros((n_beams, len(PSI))); dep = np.zeros(n_beams)
        Pf = np.zeros(n); Pd = np.zeros(n); npts = np.zeros(n, dtype=np.int32); st = np.zeros(n, dtype=np.int32)
        cnt = _lib.TorjCounters()
        _lib.check(L.torj_bundle_results(bh, dp(prof), dp(dep), dp(Pf), dp(Pd), ip(npts), ip(st), C.byref(cnt)))
        u = np.zeros((7, n))
        _lib.check(L.torj_bundle_final_state(bh, dp(u), None, None, None))
        ts = np.zeros((count, mp)); txyz = np.zeros((count, 3, mp)); tP = np.zeros((count, mp))
        _lib.check(L.torj_bundle_trajectories(bh, dp(ts), dp(txyz), dp(tP), None, None))
    finally:
        L.torj_bundle_destroy(bh)
    r = dict(dP_dV=prof, deposited_power=dep, P_final=Pf, P_deposited_ray=Pd, n_points=npts, status=st,
             counters=cnt.as_dict(), u_final=u, traj_s=ts, traj_xyz=txyz, traj_P=tP, window=window)
    check_alone(r, w, opt, window, beam_id)
    return r


def check_alone(r, w, opt, window, beam_id):
    """Invariants of one run: the counted rays are the rays without a fatal status; each beam's deposited power is the
    weighted sum of its rays' P_deposited_ray (summation order aside); consecutive samples of a trajectory never lie
    further apart than dtmax (after the vacuum leg to the plasma entry), which a skipped segment would break."""
    st = r["status"]
    ok = ~fatal(st)
    assert r["counters"]["n_rays_ok"] == int(ok.sum())
    bid = np.zeros(len(w), dtype=int) if beam_id is None else np.asarray(beam_id)
    for q in range(len(r["deposited_power"])):
        sel = ok & (bid == q)
        ref = float(np.sum(w[sel] * r["P_deposited_ray"][sel]))
        assert abs(r["deposited_power"][q] - ref) <= 1e-12 * abs(ref) + 1e-300, (q, r["deposited_power"][q], ref)
    first, count = window
    for i in range(count):
        m = min(int(r["n_points"][first + i]), r["traj_s"].shape[1])
        if m > 2:
            gap = np.diff(r["traj_s"][i, 1:m]).max()
            assert gap <= opt.dtmax * (1 + 1e-9), (first + i, gap)


def same_rays(a, b):
    for k in ("status", "n_points", "P_final", "P_deposited_ray"):
        assert np.array_equal(a[k], b[k]), k
    assert np.array_equal(a["u_final"], b["u_final"], equal_nan=True)
    for i in range(len(a["traj_s"])):  # the window's rays up to their last sample (the buffers are not cleared beyond)
        m = max(0, min(int(a["n_points"][a["window"][0] + i]), a["traj_s"].shape[1]))
        for k in ("traj_s", "traj_xyz", "traj_P"):
            assert np.array_equal(a[k][i, ..., :m], b[k][i, ..., :m]), (k, i)
    for k in ("n_acc", "n_rej", "n_rhs", "n_rays_ok"):
        assert a["counters"][k] == b["counters"][k], k
    assert np.linalg.norm(a["dP_dV"] - b["dP_dV"]) <= 1e-12 * np.linalg.norm(b["dP_dV"])
    assert np.abs(a["deposited_power"] - b["deposited_power"]).max() <= 1e-12 * np.abs(b["deposited_power"]).max()


def beam(launcher, n_rays):
    """the 1 025-ray beam (N_rings = 7, 20 azimuthal points), or the first n_rays of a 4 151-ray one (14, 20)"""
    rings = 7 if n_rays == 1025 else 14
    pos, dirs, w = tj.launch_peripheral_rays(launcher["x0"], launcher["N0"], launcher["spot"], launcher["inv_Rc"], launcher["f"],
                                             N_rings=rings, min_azimuthal_points=20)
    assert len(w) >= n_rays
    return pos[:n_rays], dirs[:n_rays], w[:n_rays]


# ------------------------------------------------------------------------------------------------------------------
# forced hand-off on bundles below the resident lanes; 16 000 segments: a hand-in every step or two
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_seg", [100, 2000, 16000])
@pytest.mark.parametrize("n_rays", [1025, 4100])
def test_forced_handoff_on_small_bundles(gpu_full, launcher, n_rays, n_seg):
    pos, dirs, w = beam(launcher, n_rays)
    window = (n_rays // 3, 3)
    for lanes in (1, 8):
        whole = run(gpu_full, pos, dirs, w, launcher["f"], 1, 1.0, tj.default_options(schedule=1, lanes_per_ray=lanes,
                                                                                     n_segments=n_seg), window)
        assert (whole["status"] == 0).all() and whole["counters"]["n_rays_ok"] == n_rays
        for sched in (2, 3):
            got = run(gpu_full, pos, dirs, w, launcher["f"], 1, 1.0, tj.default_options(schedule=sched, lanes_per_ray=lanes,
                                                                                       n_segments=n_seg), window)
            same_rays(got, whole)


def test_16000_segments_against_the_oracle(gpu_full, oracle_full, gl24, launcher):
    """64 rays of the 1 025-ray beam under the hand-off with 16 000 segments: the oracle with the same options takes the same
    steps and ends at the same power."""
    pos, dirs, w = beam(launcher, 1025)
    opt = tj.default_options(schedule=2, lanes_per_ray=1, n_segments=16000)
    got = run(gpu_full, pos, dirs, w, launcher["f"], 1, 1.0, opt, (0, 1))
    pick = np.linspace(0, len(w) - 1, 64).astype(int)
    ref = oracle_full.trace_bundle(pos[pick], dirs[pick], w[pick], launcher["f"], 1, 1.0, PSI, gl24,
                                   opts=O.OracleOptions.default(n_segments=16000), deposition="streaming")
    assert np.array_equal(got["n_points"][pick], ref["n_points"])
    assert np.abs(got["P_final"][pick] - ref["P_final"]).max() <= 1e-12


# ------------------------------------------------------------------------------------------------------------------
# life-ordered rounds over rays of very different lives: void items at the head of rounds and after retirement
# ------------------------------------------------------------------------------------------------------------------
def test_life_ordered_rounds_with_very_different_lives(gpu_full, launcher):
    """65 543 rays in blocks of 64: a third fail at initialisation (launch points off the grid), a third are 140 GHz O-mode
    rays that cross the plasma with little absorption and leave it (~1.8 m), the rest 95 / 110 GHz X-mode rays absorbed
    within ~0.4 / 0.7 m. The predicted lives differ block by block, so the queue runs over void items at the head of the
    rounds and over those of retired rays while the long rays hand in."""
    pos, dirs, w = tj.launch_peripheral_rays(launcher["x0"], launcher["N0"], launcher["spot"], launcher["inv_Rc"], launcher["f"],
                                             N_rings=66, min_azimuthal_points=14)
    n = len(w)
    kind = (np.arange(n) // 64) % 3
    pos = pos.copy()
    pos[kind == 0] = [9.0, 0.0, 0.0]
    f = np.where(kind == 1, 140e9, np.where(np.arange(n) % 2 == 0, 95e9, 110e9))
    mode = np.where(kind == 1, -1, 1)
    window = (124, 8)  # 4 O-mode rays, then 4 X-mode rays
    whole = run(gpu_full, pos, dirs, w, f, mode, 3.0, tj.default_options(schedule=1, lanes_per_ray=1), window)
    st = whole["status"]
    assert (st[kind == 0] == 2).all() and (st[kind > 0] == 0).all()
    npts = whole["n_points"]
    assert npts[kind == 1].min() > npts[kind == 2].max()
    assert npts[kind == 1].max() < 2 + 100 * 300 and whole["P_final"][kind == 1].min() > 0.5  # left before s_max, little absorbed
    L = tj.lib()
    ctx = _lib.context()
    for sched in (0, 2, 3):
        n0 = L.torj_ctx_launch_count(ctx)
        got = run(gpu_full, pos, dirs, w, f, mode, 3.0, tj.default_options(schedule=sched, lanes_per_ray=1), window)
        assert L.torj_ctx_launch_count(ctx) - n0 == (3 if sched == 3 else 4)  # + the pilot march of the life-ordered rounds
        same_rays(got, whole)


# ------------------------------------------------------------------------------------------------------------------
# warm model (plain rounds) and a plasma set under forced hand-off
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("lanes", [1, 32])
def test_warm_model_handoff(launcher, lanes):
    arr = tj.solovev_arrays(129, 129)
    arr["Te_prof"] = 15e3 * (1.0 - arr["psi_prof"]) ** 2 + 50.0
    pl = tj.Plasma(*arr.values())
    pos, dirs, w = tj.launch_peripheral_rays(launcher["x0"], launcher["N0"], launcher["spot"], launcher["inv_Rc"], 170e9,
                                             N_rings=2, min_azimuthal_points=3)
    runs = [run(pl, pos, dirs, w, 170e9, 1, 0.35, tj.default_options(absorption_model=1, schedule=s, lanes_per_ray=lanes,
                                                                     n_segments=2000), (0, 2)) for s in (1, 2)]
    assert (runs[0]["status"] == 0).all() and runs[0]["deposited_power"][0] > 0.01
    same_rays(runs[1], runs[0])


def test_plasma_set_under_forced_handoff(arrays_small, launcher):
    """two plasmas (the base case and a third of its density), one 46-ray beam through each"""
    low = dict(arrays_small, ne_prof=arrays_small["ne_prof"] * 0.3)
    pls = [tj.Plasma(*arrays_small.values()), tj.Plasma(*low.values())]
    pos, dirs, w = tj.launch_peripheral_rays(launcher["x0"], launcher["N0"], launcher["spot"], launcher["inv_Rc"], launcher["f"])
    n = len(w)
    P, D, W = np.tile(pos, (2, 1)), np.tile(dirs, (2, 1)), np.tile(w, 2)
    bid = np.repeat(np.arange(2, dtype=np.int32), n)
    for lanes in (1, 8):
        runs = [run(pls, P, D, W, launcher["f"], 1, 0.8, tj.default_options(schedule=s, lanes_per_ray=lanes, n_segments=2000),
                    (n - 2, 4), beam_id=bid, n_beams=2, beam_plasma=[0, 1]) for s in (1, 2)]
        assert (runs[0]["status"] == 0).all()
        prof = runs[0]["dP_dV"]
        assert np.linalg.norm(prof[0] - prof[1]) > 1e-3 * np.linalg.norm(prof[0])  # the plasmas do differ
        same_rays(runs[1], runs[0])


# ------------------------------------------------------------------------------------------------------------------
# n_segments above the hand-off's 16 000
# ------------------------------------------------------------------------------------------------------------------
def test_more_segments_than_the_handoff_takes(gpu_full, launcher):
    """n_segments = 20 000 on 40 000 rays, more than the resident lanes: the automatic schedule traces whole rays (no pilot
    march) and equals schedule 1; schedules 2 and 3 are refused with a message naming the limit."""
    pos, dirs, w = tj.launch_peripheral_rays(launcher["x0"], launcher["N0"], launcher["spot"], launcher["inv_Rc"], launcher["f"],
                                             N_rings=66, min_azimuthal_points=14)
    pos, dirs, w = pos[:40000], dirs[:40000], w[:40000]
    L = tj.lib()
    ctx = _lib.context()
    window = (20000, 2)
    whole = run(gpu_full, pos, dirs, w, launcher["f"], 1, 0.5, tj.default_options(schedule=1, lanes_per_ray=1, n_segments=20000),
                window)
    n0 = L.torj_ctx_launch_count(ctx)
    auto = run(gpu_full, pos, dirs, w, launcher["f"], 1, 0.5, tj.default_options(schedule=0, lanes_per_ray=1, n_segments=20000),
               window)
    assert L.torj_ctx_launch_count(ctx) - n0 == 3
    assert (whole["status"] == 0).all()
    same_rays(auto, whole)
    for sched in (2, 3):
        with pytest.raises(_lib.TorjError, match="16000"):
            tj.trace_bundle(gpu_full, pos[:32], dirs[:32], w[:32], launcher["f"], 1, 0.5, PSI,
                            options=tj.default_options(schedule=sched, n_segments=20000))
