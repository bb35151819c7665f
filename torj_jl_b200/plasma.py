"""Host-side mirror of the reference's `Plasma` (src/plasma.jl:2-58): same positional arguments, same construction
rules; the tables live in HBM after the first use.  Evaluation (src/plasma.jl:61-89) happens on the device."""
from __future__ import annotations

import ctypes as C

import numpy as np
from scipy.interpolate import CubicSpline

from . import _lib
from ._lib import _p, c_vp


def _prefilter_2d(data_rz: np.ndarray) -> np.ndarray:
    """cubic_spline_interpolation((r,z), data) coefficients (src/plasma.jl:36): data [nR,nZ] ->
    (nZ+2, nR+2) C-order == (nR+2)x(nZ+2) R-fastest."""
    nR, nZ = data_rz.shape
    buf = np.ascontiguousarray(data_rz.T, dtype=np.float64)
    out = np.empty((nZ + 2, nR + 2))
    _lib.check(_lib.lib().torj_bspline_prefilter_2d(nR, nZ, _p(buf), _p(out)))
    return out


def _prefilter_1d(y: np.ndarray) -> np.ndarray:
    y = np.ascontiguousarray(y, dtype=np.float64)
    out = np.empty(len(y) + 2)
    _lib.check(_lib.lib().torj_bspline_prefilter_1d(len(y), _p(y), _p(out)))
    return out


def _eval_1d_line(coef: np.ndarray, x0: float, h: float, n: int, x: np.ndarray) -> np.ndarray:
    """1-D cubic B-spline with Line extrapolation (Interpolations.jl semantics, SURVEY.md A.1)."""
    xl = x0 + h * (n - 1)
    xc = np.clip(x, x0, xl)
    u = (xc - x0) / h + 1.0
    i = np.clip(np.floor(u).astype(np.int64), 1, n - 1)
    d = u - i
    e = 1.0 - d
    w = [e**3 / 6.0, 2.0 / 3.0 - d**2 + d**3 / 2.0, 2.0 / 3.0 - e**2 + e**3 / 2.0, d**3 / 6.0]
    dw = [-e**2 / 2.0 / h, (-2.0 * d + 1.5 * d**2) / h, (2.0 * e - 1.5 * e**2) / h, d**2 / 2.0 / h]
    v = sum(w[k] * coef[i - 1 + k] for k in range(4))
    dv = sum(dw[k] * coef[i - 1 + k] for k in range(4))
    return v + (x - xc) * dv


def _resample_uniform(x: np.ndarray, y: np.ndarray):
    """IMAS.interp1d(x, y, :cubic).(range(x[1], x[end], length(x))) — natural cubic spline (src/plasma.jl:17-18,42-43)."""
    xr = np.linspace(x[0], x[-1], len(x))
    return xr, CubicSpline(x, y, bc_type="natural")(xr)


class Plasma:
    """Plasma(R_coords, Z_coords, psi_norm_data, psi_prof, ne_prof, Te_prof, Br_data, Bz_data, Bphi_data,
    eqt1d_psi_norm, eqt1d_volume) — reference src/plasma.jl:30-32. 2-D arrays are [nR, nZ]."""

    def __init__(self, R_coords, Z_coords, psi_norm_data, psi_prof, ne_prof, Te_prof, Br_data, Bz_data, Bphi_data,
                 eqt1d_psi_norm, eqt1d_volume, *, build="host"):
        """build="host": coefficient tables prefiltered on the host and uploaded (torj_plasma_create);
        build="device": raw arrays uploaded, prefilter + packing run on the GPU (torj_plasma_create_from_data)."""
        f8 = lambda a: np.asarray(a, dtype=np.float64)
        if build not in ("host", "device"):
            raise ValueError("build must be 'host' or 'device'")
        self.build = build
        self._raw = dict(psi=f8(psi_norm_data), psi_prof=f8(psi_prof), ne=f8(ne_prof), Te=f8(Te_prof), BR=f8(Br_data),
                         BZ=f8(Bz_data), Bphi=f8(Bphi_data), psi1d=f8(eqt1d_psi_norm), vol1d=f8(eqt1d_volume))
        self.R_coords, self.Z_coords = f8(R_coords), f8(Z_coords)
        psi_norm_data = f8(psi_norm_data)
        nR, nZ = len(self.R_coords), len(self.Z_coords)
        if psi_norm_data.shape != (nR, nZ):
            raise ValueError(f"psi_norm_data must be [nR={nR}, nZ={nZ}]")
        self._coefs = None  # the six host prefilters run on first use only: build="device" never needs them
        pr, vol = _resample_uniform(f8(eqt1d_psi_norm), f8(eqt1d_volume))  # src/plasma.jl:42-44
        self.vol_coef = _prefilter_1d(vol)
        self.vol_psi0, self.vol_dpsi, self.n_vol = float(pr[0]), float((pr[-1] - pr[0]) / (len(pr) - 1)), len(pr)
        self.psi_prof_max = float(np.max(psi_prof))  # src/plasma.jl:57
        self._handles = {}

    @property
    def coefs(self):
        """The six (nR+2)x(nZ+2) coefficient tables of src/plasma.jl:36-41, prefiltered on the host (lazily)."""
        if self._coefs is None:
            r = self._raw
            self._coefs = {"psi": _prefilter_2d(r["psi"]),
                           "lnne": self._make_2d_prof_spline(r["psi_prof"], r["ne"], r["psi"]),
                           "lnTe": self._make_2d_prof_spline(r["psi_prof"], r["Te"], r["psi"]),
                           "BR": _prefilter_2d(r["BR"]), "BZ": _prefilter_2d(r["BZ"]), "Bphi": _prefilter_2d(r["Bphi"])}
        return self._coefs

    @staticmethod
    def _make_2d_prof_spline(psi, prof, psi_norm_data):
        """reference src/plasma.jl:16-22: 1-D spline of log(profile) on a uniform psi range, evaluated (with Line
        extrapolation) at every psi_N grid node, then 2-D spline of that."""
        pr, prof2 = _resample_uniform(psi, prof)
        c1 = _prefilter_1d(np.log(prof2))
        h = (pr[-1] - pr[0]) / (len(pr) - 1)
        data = _eval_1d_line(c1, pr[0], h, len(pr), psi_norm_data)
        return _prefilter_2d(data)

    def volume(self, psi):
        """plasma.volume_psi_spline(psi) — src/plasma.jl:109,113 (host evaluation of the 1-D spline)."""
        return _eval_1d_line(self.vol_coef, self.vol_psi0, self.vol_dpsi, self.n_vol, np.asarray(psi, dtype=np.float64))

    def handle(self, ctx=None):
        """Device-resident tables for a context (uploaded once)."""
        ctx = ctx or _lib.context()
        key = ctx.value
        if key not in self._handles:
            g = _lib.TorjGrid(len(self.R_coords), len(self.Z_coords), self.R_coords[0], self.R_coords[-1],
                              self.Z_coords[0], self.Z_coords[-1])
            h = c_vp()
            if self.build == "device":
                r = self._raw
                t = lambda a: np.ascontiguousarray(a.T)  # [nR, nZ] -> R fastest
                keep = [t(r["psi"]), t(r["BR"]), t(r["BZ"]), t(r["Bphi"])]
                _lib.check(_lib.lib().torj_plasma_create_from_data(
                    ctx, C.byref(g), _p(keep[0]), _p(np.ascontiguousarray(r["psi_prof"])), _p(np.ascontiguousarray(r["ne"])),
                    _p(np.ascontiguousarray(r["Te"])), len(r["psi_prof"]), _p(keep[1]), _p(keep[2]), _p(keep[3]),
                    _p(np.ascontiguousarray(r["psi1d"])), _p(np.ascontiguousarray(r["vol1d"])), len(r["psi1d"]), C.byref(h)))
            else:
                c = self.coefs
                _lib.check(_lib.lib().torj_plasma_create(ctx, C.byref(g), _p(c["psi"]), _p(c["lnne"]), _p(c["lnTe"]), _p(c["BR"]),
                                                         _p(c["BZ"]), _p(c["Bphi"]), _p(self.vol_coef), self.n_vol, self.vol_psi0,
                                                         self.vol_dpsi, self.psi_prof_max, C.byref(h)))
            self._handles[key] = h
        return self._handles[key]

    def __del__(self):
        try:
            for h in self._handles.values():
                _lib.lib().torj_plasma_destroy(h)
            self._handles = {}
        except Exception:
            pass

    # ---- device probes (reference src/plasma.jl:61-89, src/dispersion.jl:7-15, src/absorption.jl:228-235) ----
    def probe(self, x, N, f, mode=1, ctx=None, options=None):
        """x, N: [n,3]. Returns dict of arrays: psi, ne, Te, B[n,3], X, Y, N_par, Lambda, alpha."""
        ctx = ctx or _lib.context()
        x = np.atleast_2d(np.asarray(x, dtype=np.float64)); N = np.atleast_2d(np.asarray(N, dtype=np.float64))
        n = x.shape[0]
        xt = np.ascontiguousarray(x.T); Nt = np.ascontiguousarray(N.T)
        out = np.empty((11, n))
        opt = options or _lib.default_options()
        _lib.check(_lib.lib().torj_probe(ctx, self.handle(ctx), C.byref(opt), n, _p(xt), _p(Nt), float(f), int(mode), _p(out)))
        return dict(psi=out[0], ne=out[1], Te=out[2], B=out[3:6].T.copy(), X=out[6], Y=out[7], N_par=out[8], Lambda=out[9],
                    alpha=out[10])

    def rhs(self, u, f, mode=1, ctx=None, options=None):
        """gradΛ!(du, u) for u [n,7] — reference src/solve.jl:85-95."""
        ctx = ctx or _lib.context()
        u = np.atleast_2d(np.asarray(u, dtype=np.float64))
        n = u.shape[0]
        ut = np.ascontiguousarray(u.T)
        du = np.empty((7, n))
        opt = options or _lib.default_options()
        _lib.check(_lib.lib().torj_rhs(ctx, self.handle(ctx), C.byref(opt), n, _p(ut), float(f), int(mode), _p(du)))
        return du.T.copy()


def evaluate_psi(plasma: Plasma, x, ctx=None):
    """evaluate(plasma.psi_norm_spline, x) — src/plasma.jl:61-65."""
    x = np.atleast_2d(np.asarray(x, dtype=np.float64))
    N = np.tile([1.0, 0.0, 0.0], (x.shape[0], 1))
    return plasma.probe(x, N, 1e11, 1, ctx)["psi"]
