"""make_ray / make_beam — mirrors of reference src/solve.jl:135-181 and :209-242, calling libtorj_cuda.so."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from ._lib import c_dp, c_ip
from .launch import launch_peripheral_rays
from .plasma import Plasma
from .synthetic import pol_tor_angles_2_vector

STATUS_TEXT = {
    1: "cut-off at the vacuum/plasma boundary (reference src/solve.jl:55-59)",
    2: "ray initialisation failed (assertions at reference src/solve.jl:32,138,141)",
    3: "ray ended outside the (R,Z) grid (informational: traced and deposited as the reference does)",
    4: "step limit reached", 5: "NaN in the ray state",
    6: "trajectory buffer too small",
}


def _p(a):
    return a.ctypes.data_as(c_dp)


def marshal_bundle(ray_positions, ray_directions, ray_weights, f, mode, psi_dP_dV, beam_id, n_beams, *, n_plasmas=1,
                   beam_plasma=None):
    """The host buffers torj_trace / torj_multi_trace take: component-major [3][n] rays (a Julia Matrix[n,3] as is),
    per-ray or scalar frequency / mode, psi levels, beam ids, and the result arrays. With a plasma set (torj_trace_plasmas)
    also the plasma of every beam, beam_plasma[n_beams] in [0, n_plasmas)."""
    pos = np.ascontiguousarray(np.asarray(ray_positions, dtype=np.float64).T)
    dr = np.ascontiguousarray(np.asarray(ray_directions, dtype=np.float64).T)
    n = pos.shape[1]
    wt = np.ascontiguousarray(ray_weights, dtype=np.float64)
    per_ray = int(np.ndim(f) > 0)
    fr = np.ascontiguousarray(np.atleast_1d(f), dtype=np.float64)
    md = np.ascontiguousarray(np.broadcast_to(np.atleast_1d(mode), fr.shape), dtype=np.int32)
    psi = np.ascontiguousarray(psi_dP_dV, dtype=np.float64)
    n_beams = int(n_beams) if beam_id is not None else 1
    bid = np.ascontiguousarray(beam_id, dtype=np.int32) if beam_id is not None else None
    if bid is not None and bid.shape != (n,):
        raise ValueError("beam_id must have one entry per ray")
    bp = None
    if beam_plasma is not None:
        bp = np.ascontiguousarray(beam_plasma, dtype=np.int32)
        if bp.shape != (n_beams,):
            raise ValueError(f"beam_plasma must have one entry per beam (n_beams = {n_beams}), got shape {bp.shape}")
        if bp.min() < 0 or bp.max() >= n_plasmas:
            raise ValueError(f"beam_plasma must lie in [0, {n_plasmas}) (one index into the plasmas per beam)")
        if n_plasmas > 1 and n_beams < 2:
            raise ValueError("several plasmas need several beams (beam_id, n_beams): a profile row belongs to one plasma")
    out = dict(prof=np.zeros((n_beams, len(psi))), dep=np.zeros(n_beams), Pf=np.zeros(n), Pd=np.zeros(n),
               npts=np.zeros(n, dtype=np.int32), st=np.zeros(n, dtype=np.int32), cnt=_lib.TorjCounters())
    return dict(pos=pos, dir=dr, n=n, w=wt, per_ray=per_ray, f=fr, mode=md, psi=psi, n_beams=n_beams, beam=bid,
                beam_plasma=bp, out=out)


def _plasma_list(plasma):
    """trace_bundle's plasma argument: a Plasma (None returned) or a non-empty sequence of them."""
    if isinstance(plasma, Plasma):
        return None
    pls = list(plasma)
    if not pls or not all(isinstance(p, Plasma) for p in pls):
        raise TypeError("plasma must be a Plasma or a non-empty sequence of Plasma")
    return pls


def _plasma_set(plasma, beam_plasma):
    """trace_bundle's plasma and beam_plasma: None for a Plasma, the list for a sequence (which needs beam_plasma)."""
    pls = _plasma_list(plasma)
    if pls is None and beam_plasma is not None:
        raise ValueError("beam_plasma needs a sequence of plasmas")
    if pls is not None and beam_plasma is None:
        raise ValueError("a sequence of plasmas needs beam_plasma (the plasma of every beam)")
    return pls


def bundle_result(m):
    o, nb = m["out"], m["n_beams"]
    return dict(dP_dV=o["prof"] if nb > 1 else o["prof"][0], deposited_power=o["dep"] if nb > 1 else float(o["dep"][0]),
                P_final=o["Pf"], P_deposited_ray=o["Pd"], n_points=o["npts"], status=o["st"], counters=o["cnt"].as_dict())


def trace_bundle(plasma, ray_positions, ray_directions, ray_weights, f, mode, s_max, psi_dP_dV, *,
                 options=None, ctx=None, trajectories=None, traj_max_pts=None, beam_id=None, n_beams=1, beam_plasma=None):
    """One torj_trace call on host buffers. trajectories: None or (first, count).
    beam_id/n_beams: rays of several beams in one bundle -> dP_dV[n_beams, n_psi], deposited_power[n_beams].
    plasma: a Plasma, or a sequence of Plasma on one (R,Z) grid with beam_plasma[n_beams] naming the plasma of every beam
    (torj_trace_plasmas; keep each beam's rays contiguous)."""
    pls = _plasma_set(plasma, beam_plasma)
    m = marshal_bundle(ray_positions, ray_directions, ray_weights, f, mode, psi_dP_dV, beam_id, n_beams,
                       n_plasmas=len(pls) if pls else 1, beam_plasma=beam_plasma)
    ctx = ctx or _lib.context()
    L = _lib.lib()
    n, psi, o = m["n"], m["psi"], m["out"]
    opt = options or _lib.default_options()
    t_first, t_count = trajectories if trajectories else (0, 0)
    if t_count and traj_max_pts is None:
        traj_max_pts = 2 + int(opt.n_segments * (np.ceil(s_max / opt.n_segments / opt.dtmax) + 8))
    tm = int(traj_max_pts or 0)
    ts = np.zeros((t_count, tm)); txyz = np.zeros((t_count, 3, tm)); tP = np.zeros((t_count, tm))
    tdP = np.zeros((t_count, tm)); tprof = np.zeros((t_count, len(psi)))
    rest = (C.byref(opt), n, _p(m["pos"]), _p(m["dir"]), _p(m["w"]), _p(m["f"]), m["mode"].ctypes.data_as(c_ip), m["per_ray"],
            float(s_max), len(psi), _p(psi), m["n_beams"], m["beam"].ctypes.data_as(c_ip) if m["beam"] is not None else None,
            _p(o["prof"]), _p(o["dep"]), _p(o["Pf"]), _p(o["Pd"]), o["npts"].ctypes.data_as(c_ip), o["st"].ctypes.data_as(c_ip),
            t_first, t_count, tm, _p(ts), _p(txyz), _p(tP), _p(tdP), _p(tprof), C.byref(o["cnt"]))
    if pls is None:
        _lib.check(L.torj_trace(ctx, plasma.handle(ctx), *rest))
    else:
        hs = (_lib.c_vp * len(pls))(*[p.handle(ctx).value for p in pls])
        _lib.check(L.torj_trace_plasmas(ctx, len(pls), hs, m["beam_plasma"].ctypes.data_as(c_ip), *rest))
    res = bundle_result(m)
    res.update(traj_s=ts, traj_xyz=txyz, traj_P=tP, traj_dP_ds=tdP, traj_dP_dV_ray=tprof)
    return res


def cylindrical_state(xyz, P):
    """R, phi, tau = -ln P of Cartesian samples (the reference's state is Cartesian, src/solve.jl:144); xyz [..., 3, n]."""
    x, y = xyz[..., 0, :], xyz[..., 1, :]
    with np.errstate(divide="ignore"):
        return np.hypot(x, y), np.arctan2(y, x), -np.log(P)


def make_ray(plasma: Plasma, x0, N_vacuum, f, mode, s_max, psi_dP_dV, *, options=None, ctx=None):
    """make_ray(plasma, x0, N_vacuum, f, mode, s_max, psi_dP_dV) -> (s, u, P_beam, dP_dV_ray, deposited_power)
    — reference src/solve.jl:135-136,180.  u is the list of positions (first two: launch point, plasma entry)."""
    r = trace_bundle(plasma, np.asarray(x0, dtype=np.float64)[None, :], np.asarray(N_vacuum, dtype=np.float64)[None, :],
                     [1.0], float(f), int(mode), s_max, psi_dP_dV, options=options, ctx=ctx, trajectories=(0, 1))
    st = int(r["status"][0])
    if st not in (0, 3):
        # the reference raises AssertionError / MethodError at src/solve.jl:32,138,141
        raise AssertionError(STATUS_TEXT.get(st, f"ray status {st}"))
    n = int(r["n_points"][0])
    s = r["traj_s"][0, :n].copy()
    u = [r["traj_xyz"][0, :, i].copy() for i in range(n)]
    return s, u, r["traj_P"][0, :n].copy(), r["traj_dP_dV_ray"][0].copy(), float(r["P_deposited_ray"][0])


def make_beam(plasma: Plasma, r, phi, z, steering_angle_tor, steering_angle_pol, spot_size, inverse_curvature_radius,
              f, mode, s_max, psi_dP_dV, *, options=None, ctx=None, **kwargs):
    """make_beam(...) -> (arc_lengths, trajectories, ray_powers, dP_dV, deposited_power, ray_weights)
    — reference src/solve.jl:209-210,241; kwargs go to launch_peripheral_rays (src/solve.jl:216-217)."""
    N0 = pol_tor_angles_2_vector(steering_angle_pol, steering_angle_tor)  # src/solve.jl:211
    x0 = np.array([r * np.cos(phi), r * np.sin(phi), z])                  # src/solve.jl:212-215
    pos, dirs, wts = launch_peripheral_rays(x0, N0, spot_size, inverse_curvature_radius, f, **kwargs)
    n = len(wts)
    res = trace_bundle(plasma, pos, dirs, wts, float(f), int(mode), s_max, psi_dP_dV, options=options, ctx=ctx,
                       trajectories=(0, n))
    bad = np.nonzero(~np.isin(res["status"], (0, 3)))[0]
    if len(bad):
        raise AssertionError(f"ray {int(bad[0])}: " + STATUS_TEXT.get(int(res['status'][bad[0]]), "failed"))
    arc, traj, powers = [], [], []
    for i in range(n):
        m = int(res["n_points"][i])
        arc.append(res["traj_s"][i, :m].copy())
        traj.append([res["traj_xyz"][i, :, k].copy() for k in range(m)])
        powers.append(res["traj_P"][i, :m].copy())
    return arc, traj, powers, res["dP_dV"], res["deposited_power"], wts


def _launcher_plasmas(plasma, launchers):
    """(plasmas or None, beam_plasma or None) of make_beams: a launcher's optional "plasma" key indexes a sequence of plasmas."""
    pls = _plasma_list(plasma)
    idx = [q.get("plasma", 0) for q in launchers]
    if pls is None:
        if any(i != 0 for i in idx):
            raise ValueError('a launcher names a "plasma" but make_beams got a single Plasma')
        return None, None
    bp = np.asarray(idx, dtype=np.int32)
    if bp.min() < 0 or bp.max() >= len(pls):
        raise ValueError(f'launcher "plasma" must lie in [0, {len(pls)})')
    return pls, bp


def _make_beams_device(plasma, launchers, s_max, psi_dP_dV, options, ctx, N_rings=3, min_azimuthal_points=5,
                       normalize_weight_sum=True):
    """Rays generated on the GPU (torj_bundle_create_from_launchers), traced and reduced there; only launcher
    parameters go in and profiles / per-ray scalars come out."""
    pls, bp = _launcher_plasmas(plasma, launchers)
    if pls is not None and len(pls) > 1 and len(launchers) < 2:
        raise ValueError("several plasmas need several launchers: a profile row belongs to one plasma")
    ctx = ctx or _lib.context()
    L = _lib.lib()
    if N_rings < 2:
        raise ValueError(f"N_rings = {N_rings} < 2 which is the minimum")
    nl = len(launchers)
    x0 = np.array([[q["r"] * np.cos(q["phi"]), q["r"] * np.sin(q["phi"]), q["z"]] for q in launchers]).T.copy()
    N0 = np.array([pol_tor_angles_2_vector(q["steering_angle_pol"], q["steering_angle_tor"]) for q in launchers]).T.copy()
    w = np.array([q["spot_size"] for q in launchers], dtype=np.float64)
    irc = np.array([q["inverse_curvature_radius"] for q in launchers], dtype=np.float64)
    f = np.array([q["f"] for q in launchers], dtype=np.float64)
    md = np.array([q["mode"] for q in launchers], dtype=np.int32)
    gx, gw = np.polynomial.hermite.hermgauss(2 * N_rings + 2)
    bh = _lib.c_vp(); n = C.c_int64()
    _lib.check(L.torj_bundle_create_from_launchers(ctx, nl, _p(x0), _p(N0), _p(w), _p(irc), _p(f), md.ctypes.data_as(c_ip),
                                                   int(N_rings), int(min_azimuthal_points), int(bool(normalize_weight_sum)),
                                                   _p(np.ascontiguousarray(gx)), _p(np.ascontiguousarray(gw)), C.byref(bh),
                                                   C.byref(n)))
    try:
        n = int(n.value)
        psi = np.ascontiguousarray(psi_dP_dV, dtype=np.float64)
        opt = options or _lib.default_options()
        if pls is None:
            _lib.check(L.torj_bundle_trace(bh, plasma.handle(ctx), C.byref(opt), float(s_max), len(psi), _p(psi)))
        else:
            hs = (_lib.c_vp * len(pls))(*[p.handle(ctx).value for p in pls])
            _lib.check(L.torj_bundle_trace_plasmas(bh, len(pls), hs, bp.ctypes.data_as(c_ip), C.byref(opt), float(s_max),
                                                   len(psi), _p(psi)))
        prof = np.zeros((nl, len(psi))); dep = np.zeros(nl)
        Pf = np.zeros(n); Pd = np.zeros(n); npts = np.zeros(n, dtype=np.int32); st = np.zeros(n, dtype=np.int32)
        cnt = _lib.TorjCounters()
        _lib.check(L.torj_bundle_results(bh, _p(prof), _p(dep), _p(Pf), _p(Pd), npts.ctypes.data_as(c_ip),
                                         st.ctypes.data_as(c_ip), C.byref(cnt)))
        wt = np.zeros(n)
        _lib.check(L.torj_bundle_rays(bh, None, None, _p(wt)))
    finally:
        L.torj_bundle_destroy(bh)
    per = n // nl
    res = dict(dP_dV=prof, deposited_power=dep, P_final=Pf, P_deposited_ray=Pd, n_points=npts, status=st,
               counters=cnt.as_dict())
    return prof, dep, [wt[i * per:(i + 1) * per] for i in range(nl)], [Pf[i * per:(i + 1) * per] for i in range(nl)], res


def make_beams(plasma, launchers, s_max, psi_dP_dV, *, options=None, ctx=None, device_launch=False, **kwargs):
    """Batched make_beam for scans: `launchers` is a sequence of dicts with the positional arguments of make_beam
    (r, phi, z, steering_angle_tor, steering_angle_pol, spot_size, inverse_curvature_radius, f, mode). All beams are
    traced in ONE device call; returns (dP_dV[n_beams, n_psi], deposited_power[n_beams], ray_weights per beam,
    P_final per beam). Equivalent to a host loop over make_beam (reference src/solve.jl:209-242) without trajectories.
    `plasma` may be a sequence of Plasma on one (R,Z) grid: a launcher's "plasma" key (default 0) picks the one its beam
    is traced through, and its profile row is normalised by that plasma's volume."""
    if device_launch:
        return _make_beams_device(plasma, launchers, s_max, psi_dP_dV, options, ctx, **kwargs)
    pls, bp = _launcher_plasmas(plasma, launchers)
    P, D, W, F, M, B = [], [], [], [], [], []
    for b, L in enumerate(launchers):
        N0 = pol_tor_angles_2_vector(L["steering_angle_pol"], L["steering_angle_tor"])
        x0 = np.array([L["r"] * np.cos(L["phi"]), L["r"] * np.sin(L["phi"]), L["z"]])
        p, d, w = launch_peripheral_rays(x0, N0, L["spot_size"], L["inverse_curvature_radius"], L["f"], **kwargs)
        P.append(p); D.append(d); W.append(w)
        F.append(np.full(len(w), float(L["f"]))); M.append(np.full(len(w), int(L["mode"]), dtype=np.int32))
        B.append(np.full(len(w), b, dtype=np.int32))
    res = trace_bundle(pls if pls is not None else plasma, np.concatenate(P), np.concatenate(D), np.concatenate(W),
                       np.concatenate(F), np.concatenate(M), s_max, psi_dP_dV, options=options, ctx=ctx,
                       beam_id=np.concatenate(B), n_beams=len(launchers), beam_plasma=bp)
    off = np.cumsum([0] + [len(w) for w in W])
    dP = np.atleast_2d(res["dP_dV"]); dep = np.atleast_1d(res["deposited_power"])
    return dP, dep, W, [res["P_final"][off[i]:off[i + 1]] for i in range(len(W))], res


def make_beam_series(plasmas, r, phi, z, steering_angle_tor, steering_angle_pol, spot_size, inverse_curvature_radius,
                     f, mode, s_max, psi_dP_dV, *, options=None, ctx=None, trajectories=None, **kwargs):
    """The reference's make_beam (src/solve.jl:209-242) of one launcher on each plasma of a sequence on one (R,Z) grid
    (time slices, an uncertainty ensemble), in ONE device call (torj_trace_plasmas). The beam's rays go in once per
    plasma, contiguous. Returns (dP_dV[n_plasmas, n_psi], deposited_power[n_plasmas], ray_weights, P_final[n_plasmas, n],
    res) where res holds the per-ray arrays over the whole bundle (plasma k's rays at [k n, (k+1) n)). No trajectories
    unless `trajectories` = (first, count) over that bundle: the window would otherwise hold n_plasmas beams."""
    def trace(*a, **k):
        return trace_bundle(*a, options=options, ctx=ctx, trajectories=trajectories, **k)

    return beam_series(trace, plasmas, r, phi, z, steering_angle_tor, steering_angle_pol, spot_size, inverse_curvature_radius,
                       f, mode, s_max, psi_dP_dV, **kwargs)


def beam_series(trace, plasmas, r, phi, z, steering_angle_tor, steering_angle_pol, spot_size, inverse_curvature_radius, f,
                mode, s_max, psi_dP_dV, **kwargs):
    """make_beam_series through `trace`, a function with trace_bundle's arguments (tj.trace_bundle, MultiGPU.trace_bundle)."""
    pls = _plasma_list(plasmas)
    if pls is None:
        pls = [plasmas]
    K = len(pls)
    N0 = pol_tor_angles_2_vector(steering_angle_pol, steering_angle_tor)
    x0 = np.array([r * np.cos(phi), r * np.sin(phi), z])
    pos, dirs, wts = launch_peripheral_rays(x0, N0, spot_size, inverse_curvature_radius, f, **kwargs)
    n = len(wts)
    res = trace(pls, np.tile(pos, (K, 1)), np.tile(dirs, (K, 1)), np.tile(wts, K), float(f), int(mode), s_max, psi_dP_dV,
                beam_id=np.repeat(np.arange(K, dtype=np.int32), n) if K > 1 else None, n_beams=K,
                beam_plasma=np.arange(K, dtype=np.int32))
    return (np.atleast_2d(res["dP_dV"]), np.atleast_1d(res["deposited_power"]), wts, res["P_final"].reshape(K, n), res)
