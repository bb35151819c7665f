"""Single-process multi-GPU front end (torj_multi_*): one call shards a bundle over all visible GPUs (contiguous ray
blocks or beams dealt round-robin) and sums the profiles with one ncclAllReduce over NVLink on the devices' buffers
(or on the host in device order: `deterministic=True`).  This is what a Julia `make_beam` on a multi-GPU box binds;
`bench.py --impl multi` times it, the default bench uses the one-process-per-GPU route."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from ._lib import c_dp, c_ip, c_vp
from . import absorption


def _p(a):
    return a.ctypes.data_as(c_dp)


class MultiGPU:
    def __init__(self, n_devices: int = 0):
        self.h = c_vp()
        _lib.check(_lib.lib().torj_multi_create(int(n_devices), C.byref(self.h)))
        self.n_devices = int(_lib.lib().torj_multi_device_count(self.h))
        self._plasmas = {}
        self.config = dict(sharding="contiguous", block_rays=1, deterministic=False)  # torj_multi_create's state

    def configure(self, sharding="contiguous", block_rays=1, deterministic=False):
        """sharding: "contiguous" | "block_cyclic" (blocks of block_rays consecutive rays — one beam — dealt round-robin);
        deterministic: host sum in device order instead of the NCCL all-reduce. `config` holds the current state."""
        code = {"contiguous": 0, "block_cyclic": 1}[sharding]
        _lib.check(_lib.lib().torj_multi_configure(self.h, code, int(block_rays), int(bool(deterministic))))
        self.config = dict(sharding=sharding, block_rays=int(block_rays), deterministic=bool(deterministic))

    @property
    def used_nccl(self) -> bool:
        return bool(_lib.lib().torj_multi_used_nccl(self.h))

    def abs_Al_init(self, N_absz: int):
        t, w = np.polynomial.legendre.leggauss(int(N_absz))
        absorption._int_absz, absorption._int_weights = t, w
        _lib.check(_lib.lib().torj_multi_abs_init(self.h, int(N_absz), _p(t), _p(w)))

    def _plasma(self, plasma):
        key = id(plasma)
        if key not in self._plasmas:
            r = plasma._raw
            g = _lib.TorjGrid(len(plasma.R_coords), len(plasma.Z_coords), plasma.R_coords[0], plasma.R_coords[-1],
                              plasma.Z_coords[0], plasma.Z_coords[-1])
            t = lambda a: np.ascontiguousarray(a.T)
            keep = [t(r["psi"]), t(r["BR"]), t(r["BZ"]), t(r["Bphi"])]
            h = c_vp()
            _lib.check(_lib.lib().torj_multi_plasma_create_from_data(
                self.h, C.byref(g), _p(keep[0]), _p(np.ascontiguousarray(r["psi_prof"])), _p(np.ascontiguousarray(r["ne"])),
                _p(np.ascontiguousarray(r["Te"])), len(r["psi_prof"]), _p(keep[1]), _p(keep[2]), _p(keep[3]),
                _p(np.ascontiguousarray(r["psi1d"])), _p(np.ascontiguousarray(r["vol1d"])), len(r["psi1d"]), C.byref(h)))
            self._plasmas[key] = (h, plasma)
        return self._plasmas[key][0]

    def trace_bundle(self, plasma, ray_positions, ray_directions, ray_weights, f, mode, s_max, psi_dP_dV, *, options=None,
                     beam_id=None, n_beams=1, beam_plasma=None):
        """Same arguments and result keys as torj_jl_b200.trace_bundle (without trajectories). A sequence of plasmas with
        beam_plasma traces beam b through plasmas[beam_plasma[b]] on whichever device holds its rays
        (torj_multi_trace_plasmas); each plasma's copies on the devices are made once and kept."""
        from .solve import _plasma_set, bundle_result, marshal_bundle
        pls = _plasma_set(plasma, beam_plasma)
        m = marshal_bundle(ray_positions, ray_directions, ray_weights, f, mode, psi_dP_dV, beam_id, n_beams,
                           n_plasmas=len(pls) if pls else 1, beam_plasma=beam_plasma)
        o, psi = m["out"], m["psi"]
        L = _lib.lib()
        opt = options or _lib.default_options()
        rest = (C.byref(opt), m["n"], _p(m["pos"]), _p(m["dir"]), _p(m["w"]), _p(m["f"]), m["mode"].ctypes.data_as(c_ip),
                m["per_ray"], float(s_max), len(psi), _p(psi), m["n_beams"],
                m["beam"].ctypes.data_as(c_ip) if m["beam"] is not None else None, _p(o["prof"]), _p(o["dep"]), _p(o["Pf"]),
                _p(o["Pd"]), o["npts"].ctypes.data_as(c_ip), o["st"].ctypes.data_as(c_ip), 0, 0, 0, None, None, None, None,
                None, C.byref(o["cnt"]))
        if pls is None:
            _lib.check(L.torj_multi_trace(self.h, self._plasma(plasma), *rest))
        else:
            hs = (c_vp * len(pls))(*[self._plasma(p).value for p in pls])
            _lib.check(L.torj_multi_trace_plasmas(self.h, len(pls), hs, m["beam_plasma"].ctypes.data_as(c_ip), *rest))
        return bundle_result(m)

    def make_beam_series(self, plasmas, r, phi, z, steering_angle_tor, steering_angle_pol, spot_size,
                         inverse_curvature_radius, f, mode, s_max, psi_dP_dV, *, options=None, **kwargs):
        """torj_jl_b200.make_beam_series over the devices (same arguments and result, without trajectories): the beam's
        rays on every plasma are whole beams dealt round-robin (block-cyclic with block_rays = rays per beam), so each
        device traces whole plasmas; `config` is restored afterwards."""
        from .solve import beam_series
        saved = dict(self.config)

        def trace(pls, pos, dirs, w, *a, **k):
            self.configure("block_cyclic", len(w) // len(pls), saved["deterministic"])
            try:
                return self.trace_bundle(pls, pos, dirs, w, *a, options=options, **k)
            finally:
                self.configure(**saved)

        return beam_series(trace, plasmas, r, phi, z, steering_angle_tor, steering_angle_pol, spot_size,
                           inverse_curvature_radius, f, mode, s_max, psi_dP_dV, **kwargs)

    def close(self):
        if self.h:
            for h, _ in self._plasmas.values():
                _lib.lib().torj_multi_plasma_destroy(h)
            self._plasmas = {}
            _lib.lib().torj_multi_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
