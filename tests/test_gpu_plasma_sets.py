"""Plasma sets: the beams of one bundle traced through several equilibria on one (R,Z) grid in one launch
(torj_bundle_trace_plasmas / torj_trace_plasmas, trace_bundle with a sequence of plasmas, make_beams with "plasma" keys,
make_beam_series, imas.plasmas_from_dd).

A ray does not depend on its neighbours or its lane, so with lanes_per_ray and schedule pinned every per-ray output of a set
equals that of a separate call on the ray's own plasma bit for bit; profiles agree to the order of their atomic sums."""
import ctypes as C

import numpy as np
import pytest

import torj_jl_b200 as tj
from oracle import torj_oracle as O
from torj_jl_b200 import _lib

pytestmark = pytest.mark.gpu

PSI = np.linspace(0.0, 1.0, 200)
PINNED = dict(lanes_per_ray=1, schedule=1)
S_MAX = 0.8


def dp(a):
    return a.ctypes.data_as(_lib.c_dp)


def ip(a):
    return a.ctypes.data_as(_lib.c_ip)


def l2rel(a, b):
    return np.linalg.norm(a - b) / np.linalg.norm(b)


def variant_arrays(n):
    """The base Solov'ev case and five variations on its grid that each move the answer: density x 0.3 (the reference's
    plasma_low_density, test/tests/setup.jl:57-58), a hotter core, another B0 (the resonance moves), twice the volume
    (per-beam dV) and a profile grid ending at psi_N = 0.97 (another psi_prof_max, so another plasma entry)."""
    base = tj.solovev_arrays(n, n)
    psi = base["psi_prof"]
    low = dict(base, ne_prof=base["ne_prof"] * 0.3)
    hot = dict(base, Te_prof=8.0e3 * (1.0 - psi) ** 2 + 50.0)
    b0 = tj.solovev_arrays(n, n, B0=2.1)
    vol = dict(base, eqt1d_volume=base["eqt1d_volume"] * 2.0)
    edge = dict(base, psi_prof=psi * 0.97)
    return [base, low, hot, b0, vol, edge]


def scaled_arrays(n, k):
    """k more plasmas on the grid of variant_arrays: density and temperature scans."""
    out = []
    for i in range(k):
        a = tj.solovev_arrays(n, n)
        out.append(dict(a, ne_prof=a["ne_prof"] * (0.4 + 0.1 * i), Te_prof=a["Te_prof"] * (0.8 + 0.05 * i)))
    return out


@pytest.fixture(scope="module", autouse=True)
def _abs_al_init():
    tj.abs_Al_init(24)


_SETS = {}


def plasma_set(n):
    if n not in _SETS:
        arrs = variant_arrays(n)
        _SETS[n] = (arrs, [tj.Plasma(*a.values()) for a in arrs])
    return _SETS[n]


@pytest.fixture(scope="module")
def beam46(launcher):
    return tj.launch_peripheral_rays(launcher["x0"], launcher["N0"], launcher["spot"], launcher["inv_Rc"], launcher["f"])


def bundle_run(plasmas, beam_plasma, pos, dirs, w, f, beam_id, n_beams, opt, s_max=S_MAX, psi=PSI):
    """One resident bundle traced through torj_bundle_trace (one Plasma) or torj_bundle_trace_plasmas (a list):
    results and the final state of every ray."""
    L = tj.lib()
    ctx = _lib.context()
    n = len(w)
    posT, dirT = np.ascontiguousarray(np.asarray(pos).T), np.ascontiguousarray(np.asarray(dirs).T)
    w = np.ascontiguousarray(w, dtype=np.float64)
    fr, md = np.array([f]), np.array([1], dtype=np.int32)
    bh = _lib.c_vp()
    _lib.check(L.torj_bundle_create(ctx, n, dp(posT), dp(dirT), dp(w), dp(fr), ip(md), 0, C.byref(bh)))
    try:
        if beam_id is not None:
            bid = np.ascontiguousarray(beam_id, dtype=np.int32)
            _lib.check(L.torj_bundle_set_beams(bh, n_beams, ip(bid)))
        if isinstance(plasmas, tj.Plasma):
            _lib.check(L.torj_bundle_trace(bh, plasmas.handle(ctx), C.byref(opt), s_max, len(psi), dp(psi)))
        else:
            hs = (_lib.c_vp * len(plasmas))(*[p.handle(ctx).value for p in plasmas])
            bp = np.ascontiguousarray(beam_plasma, dtype=np.int32)
            _lib.check(L.torj_bundle_trace_plasmas(bh, len(plasmas), hs, ip(bp), C.byref(opt), s_max, len(psi), dp(psi)))
        nb = n_beams if beam_id is not None else 1
        prof = np.zeros((nb, len(psi))); dep = np.zeros(nb)
        Pf = np.zeros(n); Pd = np.zeros(n); npts = np.zeros(n, dtype=np.int32); st = np.zeros(n, dtype=np.int32)
        _lib.check(L.torj_bundle_results(bh, dp(prof), dp(dep), dp(Pf), dp(Pd), ip(npts), ip(st), None))
        u = np.zeros((7, n))
        _lib.check(L.torj_bundle_final_state(bh, dp(u), None, None, None))
    finally:
        L.torj_bundle_destroy(bh)
    return dict(dP_dV=prof, deposited_power=dep, P_final=Pf, P_deposited_ray=Pd, n_points=npts, status=st, u_final=u)


def same_rays(a, ia, b, ib):
    """per-ray outputs of rays ia of result a and ib of result b are bit-identical"""
    for k in ("status", "n_points", "P_final", "P_deposited_ray"):
        assert np.array_equal(a[k][ia], b[k][ib]), k
    if "u_final" in a and "u_final" in b:
        assert np.array_equal(a["u_final"][:, ia], b["u_final"][:, ib], equal_nan=True)


def stacked(pos, dirs, w, K):
    n = len(w)
    return np.tile(pos, (K, 1)), np.tile(dirs, (K, 1)), np.tile(w, K), np.repeat(np.arange(K, dtype=np.int32), n)


# ------------------------------------------------------------------------------------------------------------------
# 1, 2, 4: one call equals K calls; the plasmas are really used; deposition against each plasma's own volume
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("grid", [65, 257])
def test_set_equals_separate_calls(grid, launcher, beam46):
    arrs, pls = plasma_set(grid)
    K = len(pls)
    pos, dirs, w = beam46
    n = len(w)
    P, D, W, B = stacked(pos, dirs, w, K)
    opt = tj.default_options(**PINNED)
    got = bundle_run(pls, np.arange(K), P, D, W, launcher["f"], B, K, opt)
    sep = [bundle_run(p, None, pos, dirs, w, launcher["f"], None, 1, opt) for p in pls]
    assert (got["status"] == 0).all()
    for k in range(K):
        same_rays(got, slice(k * n, (k + 1) * n), sep[k], slice(None))
        assert np.abs(got["dP_dV"][k] - sep[k]["dP_dV"][0]).max() <= 1e-12 * np.abs(sep[k]["dP_dV"][0]).max()
        assert abs(got["deposited_power"][k] - sep[k]["deposited_power"][0]) <= 1e-12 * sep[k]["deposited_power"][0]
    # 2: every beam's answer differs from every other plasma's by far more than the tolerances above
    for k in range(K):
        for j in range(K):
            if j != k:
                assert l2rel(got["dP_dV"][k], sep[j]["dP_dV"][0]) > 1e-4, (k, j)
    # 4: sum dV dP/dV = deposited power, each beam with its own plasma's volume (reference test/tests/test_make_beam.jl (c))
    for k in range(K):
        dV = pls[k].volume(PSI[1:]) - pls[k].volume(PSI[:-1])
        assert abs(float(np.sum(dV * got["dP_dV"][k][:-1])) - got["deposited_power"][k]) < 1e-3
    # automatic lanes and schedule: the same steps, P_final to the lane-width tolerance
    auto = tj.trace_bundle(pls, P, D, W, launcher["f"], 1, S_MAX, PSI, beam_id=B, n_beams=K, beam_plasma=np.arange(K))
    assert np.array_equal(auto["n_points"], got["n_points"])
    assert np.abs(auto["P_final"] - got["P_final"]).max() < 1e-10


def test_trajectory_window_across_two_plasmas(launcher, beam46):
    arrs, pls = plasma_set(65)
    pos, dirs, w = beam46
    n = len(w)
    P, D, W, B = stacked(pos, dirs, w, 2)
    opt = tj.default_options(**PINNED)
    got = tj.trace_bundle(pls[3:5], P, D, W, launcher["f"], 1, S_MAX, PSI, options=opt, beam_id=B, n_beams=2,
                          beam_plasma=[0, 1], trajectories=(n - 2, 4))
    a = tj.trace_bundle(pls[3], pos, dirs, w, launcher["f"], 1, S_MAX, PSI, options=opt, trajectories=(n - 2, 2),
                        traj_max_pts=got["traj_s"].shape[1])
    b = tj.trace_bundle(pls[4], pos, dirs, w, launcher["f"], 1, S_MAX, PSI, options=opt, trajectories=(0, 2),
                        traj_max_pts=got["traj_s"].shape[1])
    same_rays(got, slice(n - 2, n + 2), dict((k, np.concatenate([a[k][n - 2:], b[k][:2]])) for k in ("status", "n_points", "P_final", "P_deposited_ray")), slice(None))
    for r, (one, i) in enumerate(((a, 0), (a, 1), (b, 0), (b, 1))):
        m = int(got["n_points"][n - 2 + r])  # samples past a ray's n_points are not written
        assert np.array_equal(got["traj_s"][r, :m], one["traj_s"][i, :m]) and np.array_equal(got["traj_P"][r, :m], one["traj_P"][i, :m])
        assert np.array_equal(got["traj_xyz"][r, :, :m], one["traj_xyz"][i, :, :m])
        assert np.array_equal(got["traj_dP_ds"][r, :m], one["traj_dP_ds"][i, :m])
    # the per-ray profile of each ray is normalised by its own plasma's volume (pls[4] has twice the volume)
    assert np.abs(got["traj_dP_dV_ray"][:2] - a["traj_dP_dV_ray"]).max() <= 1e-12 * np.abs(a["traj_dP_dV_ray"]).max()
    assert np.abs(got["traj_dP_dV_ray"][2:] - b["traj_dP_dV_ray"]).max() <= 1e-12 * np.abs(b["traj_dP_dV_ray"]).max()


# ------------------------------------------------------------------------------------------------------------------
# 3: against the oracle
# ------------------------------------------------------------------------------------------------------------------
def test_set_against_oracle(launcher, beam46, gl24):
    arrs, pls = plasma_set(65)
    K = len(pls)
    pos, dirs, w = beam46
    n = len(w)
    P, D, W, B = stacked(pos, dirs, w, K)
    pick = [0, 17, 40]
    win = (0, K * n)
    got = tj.trace_bundle(pls, P, D, W, launcher["f"], 1, S_MAX, PSI, beam_id=B, n_beams=K, beam_plasma=np.arange(K),
                          trajectories=win)
    for k in range(K):
        opl = O.OraclePlasma(*arrs[k].values())
        ref = opl.trace_bundle(pos, dirs, w, launcher["f"], 1, S_MAX, PSI, gl24)
        assert abs(got["deposited_power"][k] - ref["deposited_power"]) <= 1e-6 * ref["deposited_power"], k
        for i in pick:
            ro = opl.make_ray(pos[i], dirs[i], launcher["f"], 1, S_MAX, PSI, gl24)
            r = k * n + i
            m = int(got["n_points"][r])
            assert m == len(ro["s"]), (k, i)
            xyz = got["traj_xyz"][r, :, :m]
            assert max(np.abs(xyz[0] - ro["x"]).max(), np.abs(xyz[2] - ro["z"]).max()) < 1e-9, (k, i)
            assert abs(got["P_final"][r] - ref["P_final"][i]) < 1e-12


# ------------------------------------------------------------------------------------------------------------------
# 5, 6: past the hand-off threshold; interleaved beams
# ------------------------------------------------------------------------------------------------------------------
def test_past_the_handoff_threshold(launcher):
    arrs = variant_arrays(65) + scaled_arrays(65, 10)
    pls = [tj.Plasma(*a.values()) for a in arrs]
    K = len(pls)
    assert K >= 16
    pos, dirs, w = tj.launch_peripheral_rays(launcher["x0"], launcher["N0"], launcher["spot"], launcher["inv_Rc"], launcher["f"],
                                             N_rings=7, min_azimuthal_points=20)
    n = len(w)
    nb = 64
    P, D, W, B = stacked(pos, dirs, w, nb)
    bp = np.arange(nb) % K
    assert len(W) > 37888
    got = tj.trace_bundle(pls, P, D, W, launcher["f"], 1, S_MAX, PSI, beam_id=B, n_beams=nb, beam_plasma=bp)
    assert (got["status"] == 0).all()
    sample = np.arange(0, n, 97)
    opt = tj.default_options(**PINNED)
    for b in (0, 5, 17, 40, 63):
        one = tj.trace_bundle(pls[bp[b]], pos[sample], dirs[sample], w[sample], launcher["f"], 1, S_MAX, PSI, options=opt)
        same_rays(got, b * n + sample, one, slice(None))
    # every beam on the same plasma gives the same profile (the hand-off and life prediction resolve each ray's plasma)
    for b in range(K, nb):
        assert l2rel(got["dP_dV"][b], got["dP_dV"][b % K]) < 1e-11


def test_interleaved_and_shuffled_beams(launcher, beam46):
    arrs, pls = plasma_set(65)
    K = len(pls)
    pos, dirs, w = tj.launch_peripheral_rays(launcher["x0"], launcher["N0"], launcher["spot"], launcher["inv_Rc"], launcher["f"],
                                             N_rings=4, min_azimuthal_points=8)
    n = len(w)
    opt = tj.default_options(**PINNED)
    sep = [tj.trace_bundle(p, pos, dirs, w, launcher["f"], 1, S_MAX, PSI, options=opt) for p in pls]
    # 32-ray blocks, one beam each, plasmas alternating block by block, then the beams in random order
    blocks = [(k, s) for s in range(0, n, 32) for k in range(K)]
    order = np.random.default_rng(7).permutation(len(blocks))
    P, D, W, B, src = [], [], [], [], []
    for beam, bi in enumerate(order):
        k, s = blocks[bi]
        idx = np.arange(s, min(s + 32, n))
        P.append(pos[idx]); D.append(dirs[idx]); W.append(w[idx]); B.append(np.full(len(idx), beam, dtype=np.int32))
        src.append((k, idx))
    bp = np.array([blocks[bi][0] for bi in order])
    for o in (opt, tj.default_options()):
        got = tj.trace_bundle(pls, np.concatenate(P), np.concatenate(D), np.concatenate(W), launcher["f"], 1, S_MAX, PSI,
                              options=o, beam_id=np.concatenate(B), n_beams=len(order), beam_plasma=bp)
        r = 0
        for k, idx in src:
            if o is opt:
                same_rays(got, slice(r, r + len(idx)), sep[k], idx)
            else:
                assert np.array_equal(got["n_points"][r:r + len(idx)], sep[k]["n_points"][idx])
                assert np.abs(got["P_final"][r:r + len(idx)] - sep[k]["P_final"][idx]).max() < 1e-10
            r += len(idx)


# ------------------------------------------------------------------------------------------------------------------
# 7, 8: warm model, higher harmonics, one plasma through the new entry point
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("extra", [dict(absorption_model=1), dict(max_harmonic=5)], ids=["warm", "harmonic5"])
def test_models_match_separate_calls(extra, launcher):
    arrs, pls = plasma_set(65)
    sub = [pls[0], pls[2], pls[3]]
    pos, dirs, w = tj.launch_peripheral_rays(launcher["x0"], launcher["N0"], launcher["spot"], launcher["inv_Rc"], launcher["f"],
                                             N_rings=2, min_azimuthal_points=3)
    n = len(w)
    P, D, W, B = stacked(pos, dirs, w, 3)
    for lanes in ((1, 32) if "absorption_model" in extra else (1, 4)):
        opt = tj.default_options(lanes_per_ray=lanes, schedule=1, **extra)
        got = bundle_run(sub, np.arange(3), P, D, W, launcher["f"], B, 3, opt, s_max=0.5)
        for k, p in enumerate(sub):
            one = bundle_run(p, None, pos, dirs, w, launcher["f"], None, 1, opt, s_max=0.5)
            same_rays(got, slice(k * n, (k + 1) * n), one, slice(None))
            assert abs(got["deposited_power"][k] - one["deposited_power"][0]) <= 1e-12 * max(one["deposited_power"][0], 1e-300)


def test_one_plasma_through_the_set_entry_point(launcher, beam46):
    arrs, pls = plasma_set(65)
    pos, dirs, w = beam46
    L = tj.lib()
    ctx = _lib.context()
    c0 = L.torj_ctx_launch_count(ctx)
    a = tj.trace_bundle(pls[1], pos, dirs, w, launcher["f"], 1, S_MAX, PSI, trajectories=(3, 2))
    c1 = L.torj_ctx_launch_count(ctx)
    b = tj.trace_bundle([pls[1]], pos, dirs, w, launcher["f"], 1, S_MAX, PSI, beam_plasma=[0], trajectories=(3, 2))
    c2 = L.torj_ctx_launch_count(ctx)
    assert c2 - c1 == c1 - c0  # the same kernels
    for k in ("status", "n_points", "P_final", "P_deposited_ray", "traj_s", "traj_xyz", "traj_P", "traj_dP_ds"):
        assert np.array_equal(a[k], b[k]), k
    assert np.abs(a["dP_dV"] - b["dP_dV"]).max() <= 1e-12 * np.abs(a["dP_dV"]).max()


# ------------------------------------------------------------------------------------------------------------------
# 9: Python and IMAS paths
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("device_launch", [False, True])
def test_make_beams_with_plasma_keys(device_launch, launcher):
    arrs, pls = plasma_set(65)
    base = dict(r=2.5, phi=0.0, z=0.4, spot_size=launcher["spot"], inverse_curvature_radius=launcher["inv_Rc"],
                steering_angle_tor=0.0, f=95e9, mode=1)
    Ls = [dict(base, steering_angle_pol=np.deg2rad(30.0), plasma=1), dict(base, steering_angle_pol=np.deg2rad(24.0), plasma=3),
          dict(base, steering_angle_pol=np.deg2rad(30.0), plasma=4), dict(base, steering_angle_pol=np.deg2rad(27.0))]
    dP, dep, W, Pf, res = tj.make_beams(pls, Ls, S_MAX, PSI, device_launch=device_launch)
    assert dP.shape == (4, len(PSI)) and (res["status"] == 0).all()
    for b, L in enumerate(Ls):
        one = tj.make_beams(pls[L.get("plasma", 0)], [dict((k, v) for k, v in L.items() if k != "plasma")], S_MAX, PSI,
                            device_launch=device_launch)
        assert np.array_equal(one[3][0], Pf[b])
        assert np.abs(one[0][0] - dP[b]).max() <= 1e-12 * np.abs(one[0][0]).max()
        assert abs(one[1][0] - dep[b]) <= 1e-12 * one[1][0]


def test_make_beam_series(launcher):
    arrs, pls = plasma_set(65)
    dP, dep, w, Pf, res = tj.make_beam_series(pls, 2.5, 0.0, 0.4, 0.0, np.deg2rad(30.0), launcher["spot"], launcher["inv_Rc"],
                                              launcher["f"], 1, S_MAX, PSI)
    assert dP.shape == (len(pls), len(PSI)) and dep.shape == (len(pls),) and Pf.shape == (len(pls), len(w)) and len(w) == 46
    for k, p in enumerate(pls):
        _, _, _, prof, d, _ = tj.make_beam(p, 2.5, 0.0, 0.4, 0.0, np.deg2rad(30.0), launcher["spot"], launcher["inv_Rc"],
                                           launcher["f"], 1, S_MAX, PSI)
        assert np.abs(prof - dP[k]).max() <= 1e-12 * np.abs(prof).max() and abs(d - dep[k]) <= 1e-12 * d


def test_plasmas_from_dd_series(launcher, beam46):
    arr = tj.solovev_arrays(65, 65)
    dd = tj.solovev_dd(arr, times=(1.0, 2.0, 3.0), ne_scale_per_slice=(1.0, 0.6, 0.3))
    pls = tj.plasmas_from_dd(dd)
    assert len(pls) == 3
    pos, dirs, w = beam46
    n = len(w)
    P, D, W, B = stacked(pos, dirs, w, 3)
    opt = tj.default_options(**PINNED)
    got = tj.trace_bundle(pls, P, D, W, launcher["f"], 1, S_MAX, PSI, options=opt, beam_id=B, n_beams=3, beam_plasma=[0, 1, 2])
    for k, t in enumerate((1.0, 2.0, 3.0)):
        one = tj.trace_bundle(tj.plasma_from_dd(dd, t), pos, dirs, w, launcher["f"], 1, S_MAX, PSI, options=opt)
        same_rays(got, slice(k * n, (k + 1) * n), one, slice(None))
    assert got["deposited_power"][0] != got["deposited_power"][2]


# ------------------------------------------------------------------------------------------------------------------
# 10: refusals
# ------------------------------------------------------------------------------------------------------------------
def test_refusals(launcher, beam46):
    arrs, pls = plasma_set(65)
    L = tj.lib()
    ctx = _lib.context()
    pos, dirs, w = beam46
    n = len(w)
    P, D, W, B = stacked(pos, dirs, w, 2)
    posT, dirT = np.ascontiguousarray(P.T), np.ascontiguousarray(D.T)
    W = np.ascontiguousarray(W)
    fr, md = np.array([95e9]), np.array([1], dtype=np.int32)
    other = tj.Plasma(*tj.solovev_arrays(65, 65, R_range=(0.5, 2.75)).values())
    bh = _lib.c_vp()
    _lib.check(L.torj_bundle_create(ctx, 2 * n, dp(posT), dp(dirT), dp(W), dp(fr), ip(md), 0, C.byref(bh)))

    def trace(plist, bp, n_pl=None):
        hs = (_lib.c_vp * max(len(plist), 1))(*[p.handle(ctx).value if p is not None else None for p in plist])
        bpa = np.ascontiguousarray(bp, dtype=np.int32) if bp is not None else None
        rc = L.torj_bundle_trace_plasmas(bh, len(plist) if n_pl is None else n_pl, hs, ip(bpa) if bpa is not None else None,
                                         None, S_MAX, len(PSI), dp(PSI))
        return rc, L.torj_last_error().decode()

    try:
        rc, msg = trace(pls[:2], [0, 1])
        assert rc != 0 and "need beams" in msg                         # two plasmas, one beam
        _lib.check(L.torj_bundle_set_beams(bh, 2, ip(np.ascontiguousarray(B))))
        rc, msg = trace(pls[:2], [0, 1], n_pl=0)
        assert rc != 0 and "n_plasmas must be >= 1" in msg
        rc, msg = trace([pls[0], None], [0, 1])
        assert rc != 0 and "plasmas[1] is NULL" in msg
        rc, msg = trace([pls[0], other], [0, 1])
        assert rc != 0 and "another (R,Z) grid" in msg
        rc, msg = trace(pls[:2], None)
        assert rc != 0 and "beam_plasma is NULL" in msg
        rc, msg = trace(pls[:2], [0, 2])
        assert rc != 0 and "beam_plasma[1] = 2 is outside [0, 2)" in msg
        rc, msg = trace(pls[:2], [0, 1])
        assert rc == 0, msg
        _lib.check(L.torj_ctx_sync(ctx))
    finally:
        L.torj_bundle_destroy(bh)
    # the one-shot entry point refuses the same way, before it touches its workspace
    with pytest.raises(_lib.TorjError, match="another \\(R,Z\\) grid"):
        tj.trace_bundle([pls[0], other], P, D, W, 95e9, 1, S_MAX, PSI, beam_id=B, n_beams=2, beam_plasma=[0, 1])
    import torch

    if torch.cuda.device_count() < 2:
        return  # a plasma on another device needs a second GPU
    ctx1 = _lib.context(1)
    far = pls[0].handle(ctx1)
    bh = _lib.c_vp()
    _lib.check(L.torj_bundle_create(ctx, 2 * n, dp(posT), dp(dirT), dp(W), dp(fr), ip(md), 0, C.byref(bh)))
    try:
        _lib.check(L.torj_bundle_set_beams(bh, 2, ip(np.ascontiguousarray(B))))
        hs = (_lib.c_vp * 2)(pls[0].handle(ctx).value, far.value)
        bp = np.array([0, 1], dtype=np.int32)
        assert L.torj_bundle_trace_plasmas(bh, 2, hs, ip(bp), None, S_MAX, len(PSI), dp(PSI)) != 0
        assert "is on device 1" in L.torj_last_error().decode()
    finally:
        L.torj_bundle_destroy(bh)
