"""Plasma sets on several GPUs in one process: torj_multi_trace_plasmas, MultiGPU.trace_bundle with a sequence of plasmas,
MultiGPU.make_beam_series. Runs on every visible GPU (one or more); checks that need a second device skip below that.

The multi-device front end builds its tables with the device constructor, so the single-device reference uses plasmas
built with build="device": then a ray's outputs do not depend on the device or the neighbours it was traced with, and
with lanes_per_ray and schedule pinned they agree bit for bit. Profiles agree to the order of their sums."""
import ctypes as C

import numpy as np
import pytest

import torj_jl_b200 as tj
from torj_jl_b200 import _lib
from torj_jl_b200.distributed import shard_range

pytestmark = pytest.mark.gpu

PSI = np.linspace(0.0, 1.0, 200)
PINNED = dict(lanes_per_ray=1, schedule=1)
S_MAX = 0.8
PER_RAY = ("status", "n_points", "P_final", "P_deposited_ray")


def dp(a):
    return a.ctypes.data_as(_lib.c_dp) if a is not None else None


def ip(a):
    return a.ctypes.data_as(_lib.c_ip) if a is not None else None


def variant_arrays(n):
    """The Solov'ev case and five variations on its grid that each move the answer: lower density, a hotter core,
    another B0, twice the volume (per-beam dV) and a profile grid ending at psi_N = 0.97 (another plasma entry)."""
    base = tj.solovev_arrays(n, n)
    psi = base["psi_prof"]
    return [base, dict(base, ne_prof=base["ne_prof"] * 0.3), dict(base, Te_prof=8.0e3 * (1.0 - psi) ** 2 + 50.0),
            tj.solovev_arrays(n, n, B0=2.1), dict(base, eqt1d_volume=base["eqt1d_volume"] * 2.0), dict(base, psi_prof=psi * 0.97)]


_SET = []


def device_set():
    if not _SET:
        _SET.extend(tj.Plasma(*a.values(), build="device") for a in variant_arrays(65))
    return _SET


@pytest.fixture(scope="module")
def mg():
    tj.abs_Al_init(24)
    m = tj.MultiGPU()
    m.abs_Al_init(24)
    yield m
    m.close()


@pytest.fixture(scope="module")
def ragged(launcher):
    """Five beams of 120, 46, 17, 30 and 5 rays on plasmas 0, 1, 2, 3, 5 (plasma 4 unused). Beam 0 holds more than half
    the rays, so under contiguous sharding device 0 traces that beam alone."""
    big = tj.launch_peripheral_rays(launcher["x0"], launcher["N0"], launcher["spot"], launcher["inv_Rc"], launcher["f"],
                                    N_rings=6, min_azimuthal_points=14)
    small = tj.launch_peripheral_rays(launcher["x0"], launcher["N0"], launcher["spot"], launcher["inv_Rc"], launcher["f"])
    assert len(big[2]) >= 120 and len(small[2]) == 46
    parts = [tuple(a[:120] for a in big), small, tuple(a[:17] for a in small), tuple(a[10:40] for a in big),
             tuple(a[-5:] for a in small)]
    pos = np.concatenate([p[0] for p in parts]); dirs = np.concatenate([p[1] for p in parts])
    w = np.concatenate([p[2] for p in parts])
    bid = np.concatenate([np.full(len(p[2]), b, dtype=np.int32) for b, p in enumerate(parts)])
    return pos, dirs, w, bid, np.array([0, 1, 2, 3, 5], dtype=np.int32)


def multi_c(m, handles, bp, pos, dirs, w, f, bid, nb, opt, window=(0, 0), tm=0, n_pl=None, one=False):
    """torj_multi_trace_plasmas (one: torj_multi_trace of handles[0]) through the C ABI, trajectory window included:
    (rc, error text, results)."""
    L = tj.lib()
    n = len(w)
    posT, dirT = np.ascontiguousarray(np.asarray(pos).T), np.ascontiguousarray(np.asarray(dirs).T)
    w = np.ascontiguousarray(w, dtype=np.float64)
    fr, md = np.array([f]), np.array([1], dtype=np.int32)
    bida = np.ascontiguousarray(bid, dtype=np.int32) if bid is not None else None
    bpa = np.ascontiguousarray(bp, dtype=np.int32) if bp is not None else None
    hs = (_lib.c_vp * max(len(handles), 1))(*[h.value if h is not None else None for h in handles])
    r = dict(dP_dV=np.zeros((nb, len(PSI))), deposited_power=np.zeros(nb), P_final=np.zeros(n), P_deposited_ray=np.zeros(n),
             n_points=np.zeros(n, dtype=np.int32), status=np.zeros(n, dtype=np.int32))
    c = window[1]
    t = dict(traj_s=np.zeros((c, tm)), traj_xyz=np.zeros((c, 3, tm)), traj_P=np.zeros((c, tm)), traj_dP_ds=np.zeros((c, tm)),
             traj_dP_dV_ray=np.zeros((c, len(PSI))))
    cnt = _lib.TorjCounters()
    rest = (C.byref(opt), n, dp(posT), dp(dirT), dp(w), dp(fr), ip(md), 0, S_MAX, len(PSI), dp(PSI), nb, ip(bida),
            dp(r["dP_dV"]), dp(r["deposited_power"]), dp(r["P_final"]), dp(r["P_deposited_ray"]), ip(r["n_points"]),
            ip(r["status"]), window[0], c, tm, dp(t["traj_s"]), dp(t["traj_xyz"]), dp(t["traj_P"]), dp(t["traj_dP_ds"]),
            dp(t["traj_dP_dV_ray"]), C.byref(cnt))
    if one:
        rc = L.torj_multi_trace(m.h, handles[0], *rest)
    else:
        rc = L.torj_multi_trace_plasmas(m.h, len(handles) if n_pl is None else n_pl, hs, ip(bpa), *rest)
    r.update(t, counters=cnt.as_dict())
    return rc, L.torj_last_error().decode(), r


def same_rays(a, b, ia=slice(None), ib=slice(None)):
    for k in PER_RAY:
        assert np.array_equal(a[k][ia], b[k][ib]), k


def close_profiles(a, b, rel=1e-12):
    for q in range(len(b["deposited_power"])):
        scale = np.abs(b["dP_dV"][q]).max()
        assert np.abs(a["dP_dV"][q] - b["dP_dV"][q]).max() <= rel * scale, q
    assert np.abs(a["deposited_power"] - b["deposited_power"]).max() <= rel * np.abs(b["deposited_power"]).max()


# ------------------------------------------------------------------------------------------------------------------
# 1, 2: bit for bit per ray against one device and against one call per plasma
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("sharding", [("contiguous", 1), ("block_cyclic", 23)], ids=["contiguous", "block_cyclic"])
def test_set_equals_single_device(sharding, mg, ragged, launcher):
    pls = device_set()
    pos, dirs, w, bid, bp = ragged
    nb = len(bp)
    opt = tj.default_options(**PINNED)
    one = tj.trace_bundle(pls, pos, dirs, w, launcher["f"], 1, S_MAX, PSI, options=opt, beam_id=bid, n_beams=nb, beam_plasma=bp)
    assert (one["status"] == 0).all()
    if sharding[0] == "contiguous" and mg.n_devices > 1:
        assert shard_range(len(w), 0, mg.n_devices)[1] <= 120  # device 0 holds beam 0 only
    res = {}
    for det in (False, True):
        mg.configure(sharding[0], sharding[1], deterministic=det)
        got = mg.trace_bundle(pls, pos, dirs, w, launcher["f"], 1, S_MAX, PSI, options=opt, beam_id=bid, n_beams=nb,
                              beam_plasma=bp)
        same_rays(got, one)
        close_profiles(got, one)
        if det:
            assert not mg.used_nccl
        res[det] = got
    close_profiles(res[False], res[True], rel=1e-13)  # NCCL against the host sum in device order
    mg.configure()


def test_set_equals_calls_per_plasma(mg, ragged, launcher):
    """Every beam really used its own plasma on every device: the set equals one MultiGPU call per plasma."""
    pls = device_set()
    pos, dirs, w, bid, bp = ragged
    opt = tj.default_options(**PINNED)
    mg.configure()
    got = mg.trace_bundle(pls, pos, dirs, w, launcher["f"], 1, S_MAX, PSI, options=opt, beam_id=bid, n_beams=len(bp),
                          beam_plasma=bp)
    for b, k in enumerate(bp):
        sel = np.nonzero(bid == b)[0]
        sep = mg.trace_bundle(pls[k], pos[sel], dirs[sel], w[sel], launcher["f"], 1, S_MAX, PSI, options=opt)
        same_rays(got, sep, sel)
        assert abs(got["deposited_power"][b] - sep["deposited_power"]) <= 1e-12 * sep["deposited_power"]
        assert np.abs(got["dP_dV"][b] - sep["dP_dV"]).max() <= 1e-12 * np.abs(sep["dP_dV"]).max()
    assert len({round(float(d), 12) for d in got["deposited_power"]}) == len(bp)


# ------------------------------------------------------------------------------------------------------------------
# 3: the trajectory window across a shard boundary
# ------------------------------------------------------------------------------------------------------------------
def test_trajectory_window_across_a_shard_boundary(mg, launcher):
    pls = device_set()
    pos, dirs, w = tj.launch_peripheral_rays(launcher["x0"], launcher["N0"], launcher["spot"], launcher["inv_Rc"], launcher["f"])
    n = len(w)
    P, D, W = np.tile(pos, (2, 1)), np.tile(dirs, (2, 1)), np.tile(w, 2)
    B = np.repeat([0, 1], n).astype(np.int32)
    bp = np.array([3, 4], dtype=np.int32)  # plasma 4 has twice the volume
    # a window over the beam boundary n and the shard boundary nearest to it
    cut = min((shard_range(2 * n, d, mg.n_devices)[1] for d in range(mg.n_devices - 1)), key=lambda c: abs(c - n), default=n)
    window = (min(cut, n) - 2, abs(cut - n) + 4)
    opt = tj.default_options(**PINNED)
    ref = tj.trace_bundle(pls, P, D, W, launcher["f"], 1, S_MAX, PSI, options=opt, beam_id=B, n_beams=2, beam_plasma=bp,
                          trajectories=window)
    tm = ref["traj_s"].shape[1]
    mg.configure()
    rc, msg, got = multi_c(mg, [mg._plasma(p) for p in pls], bp, P, D, W, launcher["f"], B, 2, opt, window, tm)
    assert rc == 0, msg
    same_rays(got, ref)
    for r in range(window[1]):
        m = int(ref["n_points"][window[0] + r])
        for k in ("traj_s", "traj_xyz", "traj_P", "traj_dP_ds"):
            assert np.array_equal(got[k][r, ..., :m], ref[k][r, ..., :m]), (k, r)
    scale = np.abs(ref["traj_dP_dV_ray"]).max()
    assert np.abs(got["traj_dP_dV_ray"] - ref["traj_dP_dV_ray"]).max() <= 1e-12 * scale
    assert set(B[window[0]:window[0] + window[1]]) == {0, 1}  # rows normalised by plasma 3's volume and by plasma 4's


# ------------------------------------------------------------------------------------------------------------------
# 4: scale, and the warm model
# ------------------------------------------------------------------------------------------------------------------
def test_large_set_with_default_options(mg, launcher):
    arrs = variant_arrays(65)
    for i in range(10):
        a = tj.solovev_arrays(65, 65)
        arrs.append(dict(a, ne_prof=a["ne_prof"] * (0.4 + 0.1 * i), Te_prof=a["Te_prof"] * (0.8 + 0.05 * i)))
    pls = [tj.Plasma(*a.values(), build="device") for a in arrs]
    K = len(pls)
    pos, dirs, w = tj.launch_peripheral_rays(launcher["x0"], launcher["N0"], launcher["spot"], launcher["inv_Rc"], launcher["f"],
                                             N_rings=7, min_azimuthal_points=20)
    n, nb = len(w), 64
    P, D, W = np.tile(pos, (nb, 1)), np.tile(dirs, (nb, 1)), np.tile(w, nb)
    B = np.repeat(np.arange(nb, dtype=np.int32), n)
    bp = (np.arange(nb) % K).astype(np.int32)
    assert K == 16 and len(W) == 65600
    mg.configure()
    got = mg.trace_bundle(pls, P, D, W, launcher["f"], 1, S_MAX, PSI, beam_id=B, n_beams=nb, beam_plasma=bp)
    ok = (got["status"] == 0) | (got["status"] == 3) | (got["status"] == 6)
    assert ok.all() and got["counters"]["n_rays_ok"] == len(W)
    for q in range(nb):
        sel = B == q
        ref = float(np.sum(W[sel] * got["P_deposited_ray"][sel]))
        assert abs(got["deposited_power"][q] - ref) <= 1e-12 * abs(ref), q
    # the counters are those of one single-device call per shard (same shard size: same lanes and schedule)
    total = dict.fromkeys(got["counters"], 0)
    for d in range(mg.n_devices):
        lo, hi = shard_range(len(W), d, mg.n_devices)
        one = tj.trace_bundle(pls, P[lo:hi], D[lo:hi], W[lo:hi], launcher["f"], 1, S_MAX, PSI, beam_id=B[lo:hi], n_beams=nb,
                              beam_plasma=bp)
        for k in total:
            total[k] += one["counters"][k]
        same_rays(got, one, slice(lo, hi))
    assert got["counters"] == total


def test_warm_model_set(mg, launcher):
    pls = device_set()
    sub = [pls[0], pls[2], pls[3]]
    pos, dirs, w = tj.launch_peripheral_rays(launcher["x0"], launcher["N0"], launcher["spot"], launcher["inv_Rc"], launcher["f"],
                                             N_rings=2, min_azimuthal_points=3)
    n = len(w)
    P, D, W = np.tile(pos, (3, 1)), np.tile(dirs, (3, 1)), np.tile(w, 3)
    B = np.repeat(np.arange(3, dtype=np.int32), n)
    opt = tj.default_options(lanes_per_ray=32, schedule=1, absorption_model=1)
    mg.configure("block_cyclic", n)
    try:
        got = mg.trace_bundle(sub, P, D, W, launcher["f"], 1, 0.5, PSI, options=opt, beam_id=B, n_beams=3, beam_plasma=[0, 1, 2])
    finally:
        mg.configure()
    one = tj.trace_bundle(sub, P, D, W, launcher["f"], 1, 0.5, PSI, options=opt, beam_id=B, n_beams=3, beam_plasma=[0, 1, 2])
    same_rays(got, one)
    close_profiles(got, one)


# ------------------------------------------------------------------------------------------------------------------
# 5: make_beam_series
# ------------------------------------------------------------------------------------------------------------------
def test_make_beam_series(mg, launcher):
    pls = device_set()
    opt = tj.default_options(**PINNED)
    args = (2.5, 0.0, 0.4, 0.0, np.deg2rad(30.0), launcher["spot"], launcher["inv_Rc"], launcher["f"], 1, S_MAX, PSI)
    mg.configure("block_cyclic", 7, deterministic=True)
    got = mg.make_beam_series(pls, *args, options=opt)
    assert mg.config == dict(sharding="block_cyclic", block_rays=7, deterministic=True)
    ref = tj.make_beam_series(pls, *args, options=opt)
    assert got[0].shape == (len(pls), len(PSI)) and got[3].shape == ref[3].shape
    assert np.array_equal(got[2], ref[2]) and np.array_equal(got[3], ref[3])
    same_rays(got[4], ref[4])
    close_profiles(got[4], ref[4])
    mg.configure()


# ------------------------------------------------------------------------------------------------------------------
# 6: refusals, each before anything is enqueued: the workspaces survive
# ------------------------------------------------------------------------------------------------------------------
def test_refusals_leave_the_workspaces(mg, ragged, launcher):
    pls = device_set()
    pos, dirs, w, bid, bp = ragged
    nb = len(bp)
    opt = tj.default_options(**PINNED)
    mg.configure("contiguous", 1, deterministic=True)
    hs = [mg._plasma(p) for p in pls]
    rc, msg, base = multi_c(mg, hs, bp, pos, dirs, w, launcher["f"], bid, nb, opt)
    assert rc == 0, msg
    other_grid = tj.Plasma(*tj.solovev_arrays(65, 65, R_range=(0.5, 2.75)).values(), build="device")
    twin = tj.MultiGPU(mg.n_devices)        # the same devices, other contexts
    single = tj.MultiGPU(1)                 # fewer devices where more than one is visible
    try:
        twin.abs_Al_init(24)
        single.abs_Al_init(24)
        foreign = twin._plasma(pls[0])
        narrow = single._plasma(pls[0])
        cases = [
            (dict(handles=hs, n_pl=0), "torj_multi_trace_plasmas: n_plasmas must be >= 1"),
            (dict(handles=hs[:1] + [None] + hs[2:]), "torj_multi_trace_plasmas: plasmas[1] is NULL"),
            (dict(handles=hs[:5] + [mg._plasma(other_grid)]), "plasmas[5] is on another (R,Z) grid"),
            (dict(handles=hs, bp=None), "torj_multi_trace_plasmas: beam_plasma is NULL"),
            (dict(handles=hs, bp=np.array([0, 1, 2, 3, 6], dtype=np.int32)), "beam_plasma[4] = 6 is outside [0, 6)"),
            (dict(handles=hs, bid=None, nb=1), "6 plasmas need beams"),
            (dict(handles=hs[:1] + [foreign] + hs[2:]), "torj_multi_trace_plasmas: plasmas[1] belongs to another torj_multi"),
        ]
        if mg.n_devices > 1:
            cases.append((dict(handles=hs[:2] + [narrow] + hs[3:]),
                          "torj_multi_trace_plasmas: plasmas[2] was created on a different device set"))
        for kw, text in cases:
            a = dict(handles=hs, bp=bp, bid=bid, nb=nb)
            a.update(kw)
            rc, msg, _ = multi_c(mg, a["handles"], a["bp"], pos, dirs, w, launcher["f"], a["bid"], a["nb"], opt,
                                 n_pl=a.get("n_pl"))
            assert rc != 0 and text in msg, (text, msg)
            rc, msg, again = multi_c(mg, hs, bp, pos, dirs, w, launcher["f"], bid, nb, opt)
            assert rc == 0, msg
            same_rays(again, base)
            close_profiles(again, base)  # the order of a device's atomic sums is not fixed
        # the one-plasma entry point refuses a foreign plasma the same way, with its own texts
        one = [(foreign, "torj_multi_trace: plasma belongs to another torj_multi")]
        if mg.n_devices > 1:
            one.append((narrow, "torj_multi_trace: plasma was created on a different device set"))
        for h, text in one:
            rc, msg, _ = multi_c(mg, [h], None, pos, dirs, w, launcher["f"], bid, nb, opt, one=True)
            assert rc != 0 and msg.startswith(text), msg
            rc, msg, again = multi_c(mg, hs, bp, pos, dirs, w, launcher["f"], bid, nb, opt)
            assert rc == 0, msg
            same_rays(again, base)
    finally:
        twin.close()
        single.close()
        mg.configure()

