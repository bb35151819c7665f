"""make_ray / make_beam — mirrors of reference src/solve.jl:135-181 and :209-242, calling libtorj_cuda.so."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from ._lib import _ip, _p, c_vp
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
    return dict(pos=pos, dir=dr, n=n, w=wt, per_ray=per_ray, f=fr, mode=md, psi=psi, n_beams=n_beams, beam=bid,
                beam_plasma=bp, out=bundle_outputs(n, n_beams, len(psi)))


def bundle_outputs(n, n_beams, n_psi):
    """The result arrays of a bundle of n rays (`out` of marshal_bundle)."""
    return dict(prof=np.zeros((n_beams, n_psi)), dep=np.zeros(n_beams), Pf=np.zeros(n), Pd=np.zeros(n),
                npts=np.zeros(n, dtype=np.int32), st=np.zeros(n, dtype=np.int32), cnt=_lib.TorjCounters())


def oneshot_args(m, opt, s_max, window=(0, 0, 0), traj=None):
    """The arguments of torj_trace / torj_multi_trace (and their _plasmas forms) after the plasma ones, for the bundle m of
    marshal_bundle, the trajectory window (first, count, max_pts) and trace_bundle's `traj` arrays (None: NULL)."""
    o, psi = m["out"], m["psi"]
    traj_bufs = [_p(a) for a in traj.values()] if traj is not None else [None] * 5
    return (C.byref(opt), m["n"], _p(m["pos"]), _p(m["dir"]), _p(m["w"]), _p(m["f"]), _ip(m["mode"]), m["per_ray"],
            float(s_max), len(psi), _p(psi), m["n_beams"], _ip(m["beam"]), _p(o["prof"]), _p(o["dep"]), _p(o["Pf"]),
            _p(o["Pd"]), _ip(o["npts"]), _ip(o["st"]), *window, *traj_bufs, C.byref(o["cnt"]))


def plasma_call(L, name, plasma, beam_plasma, handle):
    """The library function of a trace through `plasma` and its plasma arguments: `name` with (handle(plasma),) for a
    Plasma; `name`_plasmas with (n_plasmas, handles, beam_plasma) for a list of them."""
    if isinstance(plasma, Plasma):
        return getattr(L, name), (handle(plasma),)
    hs = (c_vp * len(plasma))(*[handle(p).value for p in plasma])
    return getattr(L, name + "_plasmas"), (len(plasma), hs, _ip(beam_plasma))


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


def device_tensor(ptr, n, typestr):
    """A torch CUDA tensor over n elements of a device buffer the library owns (no copy; torch finds the device from the
    pointer). It is valid only as long as that buffer."""
    import torch

    class _DevBuf:
        __cuda_array_interface__ = {"shape": (int(n),), "typestr": typestr, "version": 2, "data": (int(ptr or 0), False)}
    return torch.as_tensor(_DevBuf())


def trace_bundle(plasma, ray_positions, ray_directions, ray_weights, f, mode, s_max, psi_dP_dV, *,
                 options=None, ctx=None, trajectories=None, traj_max_pts=None, beam_id=None, n_beams=1, beam_plasma=None,
                 exact_sum=False, reduce_exact=None):
    """One torj_trace call on host buffers. trajectories: None or (first, count).
    beam_id/n_beams: rays of several beams in one bundle -> dP_dV[n_beams, n_psi], deposited_power[n_beams].
    plasma: a Plasma, or a sequence of Plasma on one (R,Z) grid with beam_plasma[n_beams] naming the plasma of every beam
    (torj_trace_plasmas; keep each beam's rays contiguous).
    exact_sum: book the profile in an exact fixed-point sum (torj_ctx_set_exact_sum), so dP_dV and deposited_power are
    bit-identical under any schedule, ray order and device count; weights |w| <= 2^40.
    reduce_exact (needs exact_sum): fn(words), called between the trace and the conversion of the profile. `words` is the
    bundle's exact accumulator as an int64 torch CUDA tensor (the library's buffer itself, torj_bundle_device_exact_words);
    fn must leave in it the word-by-word integer sum over every process that traced a part of the bundle (an all-reduce
    with SUM; distributed.trace_sharded(..., exact_sum=True) passes one). dP_dV and deposited_power are then the profile of
    the summed words: the bits of one trace of all the processes' rays, at a fixed lanes_per_ray. The result also holds
    `sum_weights` (of the sum; per beam when n_beams > 1) and `local_vector`, this process's own converted vector
    [n_beams][n_psi | deposited | sum w]."""
    if reduce_exact is not None and not exact_sum:
        raise ValueError("reduce_exact needs exact_sum=True: only the exact accumulator sums across processes without rounding")
    pls = _plasma_set(plasma, beam_plasma)
    m = marshal_bundle(ray_positions, ray_directions, ray_weights, f, mode, psi_dP_dV, beam_id, n_beams,
                       n_plasmas=len(pls) if pls else 1, beam_plasma=beam_plasma)
    ctx = ctx or _lib.context()
    L = _lib.lib()
    _lib.check(L.torj_ctx_set_exact_sum(ctx, int(bool(exact_sum))))
    opt = options or _lib.default_options()
    t_first, t_count = trajectories if trajectories else (0, 0)
    if t_count and traj_max_pts is None:
        traj_max_pts = 2 + int(opt.n_segments * (np.ceil(s_max / opt.n_segments / opt.dtmax) + 8))
    tm = int(traj_max_pts or 0)
    window = (t_first, t_count, tm)
    ts = np.zeros((t_count, tm)); txyz = np.zeros((t_count, 3, tm)); tP = np.zeros((t_count, tm))
    tdP = np.zeros((t_count, tm)); tprof = np.zeros((t_count, len(m["psi"])))
    traj = dict(traj_s=ts, traj_xyz=txyz, traj_P=tP, traj_dP_ds=tdP, traj_dP_dV_ray=tprof)
    if reduce_exact is not None:
        bh = c_vp()
        _lib.check(L.torj_bundle_create(ctx, m["n"], _p(m["pos"]), _p(m["dir"]), _p(m["w"]), _p(m["f"]), _ip(m["mode"]),
                                        m["per_ray"], C.byref(bh)))
        return _trace_resident(ctx, bh, m, pls or plasma, m["beam_plasma"], opt, s_max, traj=traj, reduce_exact=reduce_exact,
                               prepare=[(L.torj_bundle_set_beams, bh, m["n_beams"], _ip(m["beam"])),
                                        (L.torj_bundle_set_window, bh, *window)])
    fn, pa = plasma_call(L, "torj_trace", pls or plasma, m["beam_plasma"], lambda p: p.handle(ctx))
    _lib.check(fn(ctx, *pa, *oneshot_args(m, opt, s_max, window, traj)))
    res = bundle_result(m)
    res.update(traj)
    return res


def _trace_resident(ctx, bh, m, plasma, beam_plasma, opt, s_max, *, prepare=(), traj=None, reduce_exact=None):
    """Trace the bundle bh that the caller has just created, and destroy it however the call ends: the library calls
    `prepare` [(fn, *args)], the trace through `plasma`, reduce_exact's sum of the exact words (see trace_bundle), then
    the results into m's arrays (ray weights too when m["out"] has "w") and the trajectories into traj's arrays."""
    L = _lib.lib()
    o, nb, psi = m["out"], m["n_beams"], m["psi"]
    res = dict(traj or {})
    try:
        for fn, *args in prepare:
            _lib.check(fn(*args))
        fn, pa = plasma_call(L, "torj_bundle_trace", plasma, beam_plasma, lambda p: p.handle(ctx))
        _lib.check(fn(bh, *pa, C.byref(opt), float(s_max), len(psi), _p(psi)))
        if reduce_exact is not None:
            import torch

            ptr, n_words = c_vp(), C.c_int64()
            _lib.check(L.torj_bundle_device_exact_words(bh, C.byref(ptr), C.byref(n_words)))
            n_vec = nb * (len(psi) + 2)
            # the library works on its context's stream, the reduction on torch's current one: each waits for the other
            _lib.check(L.torj_ctx_sync(ctx))
            local_vector = device_tensor(L.torj_bundle_device_profile(bh), n_vec, "<f8").cpu().numpy()
            words = device_tensor(ptr.value, n_words.value, "<i8")
            reduce_exact(words)
            if words.is_cuda:
                torch.cuda.current_stream(words.device).synchronize()
            _lib.check(L.torj_bundle_finalize_exact(bh))
        _lib.check(L.torj_bundle_results(bh, _p(o["prof"]), _p(o["dep"]), _p(o["Pf"]), _p(o["Pd"]), _ip(o["npts"]),
                                         _ip(o["st"]), C.byref(o["cnt"])))
        if "w" in o:
            _lib.check(L.torj_bundle_rays(bh, None, None, _p(o["w"])))
        if traj is not None and len(traj["traj_s"]):
            _lib.check(L.torj_bundle_trajectories(bh, *(_p(a) for a in traj.values())))
        if reduce_exact is not None:
            vec = device_tensor(L.torj_bundle_device_profile(bh), n_vec, "<f8").cpu().numpy()
            res.update(sum_weights=_lib.split_profile_vector(vec, nb)[2], local_vector=local_vector)
    finally:
        L.torj_bundle_destroy(bh)
    return {**bundle_result(m), **res}


def cylindrical_state(xyz, P):
    """R, phi, tau = -ln P of Cartesian samples (the reference's state is Cartesian, src/solve.jl:144); xyz [..., 3, n]."""
    x, y = xyz[..., 0, :], xyz[..., 1, :]
    with np.errstate(divide="ignore"):
        return np.hypot(x, y), np.arctan2(y, x), -np.log(P)


def make_ray(plasma: Plasma, x0, N_vacuum, f, mode, s_max, psi_dP_dV, *, options=None, ctx=None, exact_sum=False):
    """make_ray(plasma, x0, N_vacuum, f, mode, s_max, psi_dP_dV) -> (s, u, P_beam, dP_dV_ray, deposited_power)
    — reference src/solve.jl:135-136,180.  u is the list of positions (first two: launch point, plasma entry).
    exact_sum: see trace_bundle."""
    r = trace_bundle(plasma, np.asarray(x0, dtype=np.float64)[None, :], np.asarray(N_vacuum, dtype=np.float64)[None, :],
                     [1.0], float(f), int(mode), s_max, psi_dP_dV, options=options, ctx=ctx, trajectories=(0, 1),
                     exact_sum=exact_sum)
    st = int(r["status"][0])
    if st not in (0, 3):
        # the reference raises AssertionError / MethodError at src/solve.jl:32,138,141
        raise AssertionError(STATUS_TEXT.get(st, f"ray status {st}"))
    n = int(r["n_points"][0])
    s = r["traj_s"][0, :n].copy()
    u = [r["traj_xyz"][0, :, i].copy() for i in range(n)]
    return s, u, r["traj_P"][0, :n].copy(), r["traj_dP_dV_ray"][0].copy(), float(r["P_deposited_ray"][0])


def launch_geometry(r, phi, z, steering_angle_tor, steering_angle_pol):
    """make_beam's launch point x0 = (r cos phi, r sin phi, z) (reference src/solve.jl:212-215) and direction N0
    (src/solve.jl:211); componentwise, so arrays of n launchers give [3, n] each."""
    return (np.array([r * np.cos(phi), r * np.sin(phi), z]),
            pol_tor_angles_2_vector(steering_angle_pol, steering_angle_tor))


GEOMETRY = ("r", "phi", "z", "steering_angle_tor", "steering_angle_pol")  # launch_geometry's keys of a launcher


def make_beam(plasma: Plasma, r, phi, z, steering_angle_tor, steering_angle_pol, spot_size, inverse_curvature_radius,
              f, mode, s_max, psi_dP_dV, *, options=None, ctx=None, exact_sum=False, **kwargs):
    """make_beam(...) -> (arc_lengths, trajectories, ray_powers, dP_dV, deposited_power, ray_weights)
    — reference src/solve.jl:209-210,241; kwargs go to launch_peripheral_rays (src/solve.jl:216-217).
    exact_sum: see trace_bundle."""
    x0, N0 = launch_geometry(r, phi, z, steering_angle_tor, steering_angle_pol)
    pos, dirs, wts = launch_peripheral_rays(x0, N0, spot_size, inverse_curvature_radius, f, **kwargs)
    n = len(wts)
    res = trace_bundle(plasma, pos, dirs, wts, float(f), int(mode), s_max, psi_dP_dV, options=options, ctx=ctx,
                       trajectories=(0, n), exact_sum=exact_sum)
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


def _make_beams_device(plasma, launchers, s_max, psi_dP_dV, options, ctx, exact_sum, N_rings=3, min_azimuthal_points=5,
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

    def col(k, dtype=np.float64):
        return np.array([q[k] for q in launchers], dtype=dtype)
    x0, N0 = launch_geometry(*map(col, GEOMETRY))
    w, irc, f, md = col("spot_size"), col("inverse_curvature_radius"), col("f"), col("mode", np.int32)
    gx, gw = np.polynomial.hermite.hermgauss(2 * N_rings + 2)
    psi = np.ascontiguousarray(psi_dP_dV, dtype=np.float64)
    bh, n = c_vp(), C.c_int64()
    _lib.check(L.torj_bundle_create_from_launchers(ctx, nl, _p(x0), _p(N0), _p(w), _p(irc), _p(f), _ip(md), int(N_rings),
                                                   int(min_azimuthal_points), int(bool(normalize_weight_sum)), _p(gx), _p(gw),
                                                   C.byref(bh), C.byref(n)))
    m = dict(out=dict(bundle_outputs(n.value, nl, len(psi)), w=np.zeros(n.value)), n_beams=nl, psi=psi)
    res = _trace_resident(ctx, bh, m, pls or plasma, bp, options or _lib.default_options(), s_max,
                          prepare=[(L.torj_ctx_set_exact_sum, ctx, int(bool(exact_sum)))])
    wt, Pf = m["out"]["w"], res["P_final"]
    # [n_launchers, n_psi] and [n_launchers] for one launcher too
    res.update(dP_dV=np.atleast_2d(res["dP_dV"]), deposited_power=np.atleast_1d(res["deposited_power"]))
    per = len(Pf) // nl
    return (res["dP_dV"], res["deposited_power"], [wt[i * per:(i + 1) * per] for i in range(nl)],
            [Pf[i * per:(i + 1) * per] for i in range(nl)], res)


def make_beams(plasma, launchers, s_max, psi_dP_dV, *, options=None, ctx=None, device_launch=False, exact_sum=False, **kwargs):
    """Batched make_beam for scans: `launchers` is a sequence of dicts with the positional arguments of make_beam
    (r, phi, z, steering_angle_tor, steering_angle_pol, spot_size, inverse_curvature_radius, f, mode). All beams are
    traced in ONE device call; returns (dP_dV[n_beams, n_psi], deposited_power[n_beams], ray_weights per beam,
    P_final per beam). Equivalent to a host loop over make_beam (reference src/solve.jl:209-242) without trajectories.
    `plasma` may be a sequence of Plasma on one (R,Z) grid: a launcher's "plasma" key (default 0) picks the one its beam
    is traced through, and its profile row is normalised by that plasma's volume. exact_sum: see trace_bundle."""
    if device_launch:
        return _make_beams_device(plasma, launchers, s_max, psi_dP_dV, options, ctx, exact_sum, **kwargs)
    pls, bp = _launcher_plasmas(plasma, launchers)
    P, D, W, F, M, B = [], [], [], [], [], []
    for b, L in enumerate(launchers):
        x0, N0 = launch_geometry(*(L[k] for k in GEOMETRY))
        p, d, w = launch_peripheral_rays(x0, N0, L["spot_size"], L["inverse_curvature_radius"], L["f"], **kwargs)
        P.append(p); D.append(d); W.append(w)
        F.append(np.full(len(w), float(L["f"]))); M.append(np.full(len(w), int(L["mode"]), dtype=np.int32))
        B.append(np.full(len(w), b, dtype=np.int32))
    res = trace_bundle(pls if pls is not None else plasma, np.concatenate(P), np.concatenate(D), np.concatenate(W),
                       np.concatenate(F), np.concatenate(M), s_max, psi_dP_dV, options=options, ctx=ctx,
                       beam_id=np.concatenate(B), n_beams=len(launchers), beam_plasma=bp, exact_sum=exact_sum)
    off = np.cumsum([0] + [len(w) for w in W])
    dP = np.atleast_2d(res["dP_dV"]); dep = np.atleast_1d(res["deposited_power"])
    return dP, dep, W, [res["P_final"][off[i]:off[i + 1]] for i in range(len(W))], res


def make_beam_series(plasmas, r, phi, z, steering_angle_tor, steering_angle_pol, spot_size, inverse_curvature_radius,
                     f, mode, s_max, psi_dP_dV, *, options=None, ctx=None, trajectories=None, exact_sum=False, **kwargs):
    """The reference's make_beam (src/solve.jl:209-242) of one launcher on each plasma of a sequence on one (R,Z) grid
    (time slices, an uncertainty ensemble), in ONE device call (torj_trace_plasmas). The beam's rays go in once per
    plasma, contiguous. Returns (dP_dV[n_plasmas, n_psi], deposited_power[n_plasmas], ray_weights, P_final[n_plasmas, n],
    res) where res holds the per-ray arrays over the whole bundle (plasma k's rays at [k n, (k+1) n)). No trajectories
    unless `trajectories` = (first, count) over that bundle: the window would otherwise hold n_plasmas beams.
    exact_sum: see trace_bundle."""
    def trace(*a, **k):
        return trace_bundle(*a, options=options, ctx=ctx, trajectories=trajectories, exact_sum=exact_sum, **k)

    return beam_series(trace, plasmas, r, phi, z, steering_angle_tor, steering_angle_pol, spot_size, inverse_curvature_radius,
                       f, mode, s_max, psi_dP_dV, **kwargs)


def beam_series(trace, plasmas, r, phi, z, steering_angle_tor, steering_angle_pol, spot_size, inverse_curvature_radius, f,
                mode, s_max, psi_dP_dV, **kwargs):
    """make_beam_series through `trace`, a function with trace_bundle's arguments (tj.trace_bundle, MultiGPU.trace_bundle)."""
    pls = _plasma_list(plasmas)
    if pls is None:
        pls = [plasmas]
    K = len(pls)
    x0, N0 = launch_geometry(r, phi, z, steering_angle_tor, steering_angle_pol)
    pos, dirs, wts = launch_peripheral_rays(x0, N0, spot_size, inverse_curvature_radius, f, **kwargs)
    n = len(wts)
    res = trace(pls, np.tile(pos, (K, 1)), np.tile(dirs, (K, 1)), np.tile(wts, K), float(f), int(mode), s_max, psi_dP_dV,
                beam_id=np.repeat(np.arange(K, dtype=np.int32), n) if K > 1 else None, n_beams=K,
                beam_plasma=np.arange(K, dtype=np.int32))
    return (np.atleast_2d(res["dP_dV"]), np.atleast_1d(res["deposited_power"]), wts, res["P_final"].reshape(K, n), res)
