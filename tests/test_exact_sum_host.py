"""Exact deposition sums, host side: the C symbols and their bindings exist, every Python entry point takes `exact_sum`
and sets the context's (or the torj_multi's) mode to it before it traces, and MultiGPU.config keeps its three keys.
The library is replaced by a recorder, so this runs without a GPU."""
import ctypes as C
import inspect

import numpy as np
import pytest

import torj_jl_b200 as tj
from torj_jl_b200 import _lib


def test_symbols_and_signatures():
    L = _lib.lib()
    for name in ("torj_ctx_set_exact_sum", "torj_multi_set_exact_sum"):
        assert hasattr(L, name)
        assert _lib.SIGNATURES[name] == (C.c_int, [_lib.c_vp, C.c_int32])
    for fn in (tj.trace_bundle, tj.make_ray, tj.make_beam, tj.make_beams, tj.make_beam_series, tj.MultiGPU.trace_bundle,
               tj.MultiGPU.make_beam_series):
        p = inspect.signature(fn).parameters["exact_sum"]
        assert p.kind is inspect.Parameter.KEYWORD_ONLY and p.default is False, fn


class Recorder:
    """Stands in for libtorj_cuda.so: every function returns 0 and is logged with its arguments."""

    def __init__(self):
        self.calls = []

    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)

        def fn(*args):
            self.calls.append((name, args))
            return 0
        return fn

    def names(self):
        return [n for n, _ in self.calls]

    def modes(self, fn):
        """(value set, whether it came before a trace call) for every set_exact_sum of the log"""
        out = []
        for i, (n, a) in enumerate(self.calls):
            if n == fn:
                traced = any("trace" in m for m in self.names()[i + 1:])
                out.append((int(a[1]), traced))
        return out


@pytest.fixture
def rec(monkeypatch):
    r = Recorder()
    monkeypatch.setattr(_lib, "lib", lambda: r)
    return r


CTX = C.c_void_p(0x1234)
PSI = np.linspace(0.0, 1.0, 12)


def _opts():
    o = _lib.TorjOptions()
    o.n_segments, o.dtmax = 100, 1e-4
    return o


def _plasmas(k):
    arr = tj.solovev_arrays(17, 17)
    return [tj.Plasma(*arr.values(), build="device") for _ in range(k)]  # host prefilters only: no device involved


LAUNCHER = dict(r=2.5, phi=0.0, z=0.4, steering_angle_tor=0.0, steering_angle_pol=0.5, spot_size=0.02,
                inverse_curvature_radius=0.25, f=95e9, mode=1)


@pytest.mark.parametrize("exact", [True, False])
def test_every_entry_point_sets_the_mode_it_was_given(rec, exact):
    pl, = _plasmas(1)
    a, b = _plasmas(2)
    beam = (2.5, 0.0, 0.4, 0.0, 0.5, 0.02, 0.25, 95e9, 1, 0.5, PSI)
    pos, dirs = np.tile([2.5, 0.0, 0.4], (4, 1)), np.tile(tj.pol_tor_angles_2_vector(0.5, 0.0), (4, 1))
    calls = {
        "trace_bundle": lambda: tj.trace_bundle(pl, pos, dirs, np.full(4, 0.25), 95e9, 1, 0.5, PSI, options=_opts(), ctx=CTX,
                                                exact_sum=exact),
        "trace_bundle set": lambda: tj.trace_bundle([a, b], pos, dirs, np.full(4, 0.25), 95e9, 1, 0.5, PSI, options=_opts(),
                                                    ctx=CTX, beam_id=[0, 0, 1, 1], n_beams=2, beam_plasma=[0, 1],
                                                    exact_sum=exact),
        "make_ray": lambda: tj.make_ray(pl, [2.5, 0.0, 0.4], tj.pol_tor_angles_2_vector(0.5, 0.0), 95e9, 1, 0.5, PSI,
                                        options=_opts(), ctx=CTX, exact_sum=exact),
        "make_beam": lambda: tj.make_beam(pl, *beam, options=_opts(), ctx=CTX, exact_sum=exact),
        "make_beams": lambda: tj.make_beams(pl, [LAUNCHER, LAUNCHER], 0.5, PSI, options=_opts(), ctx=CTX, exact_sum=exact),
        "make_beams device": lambda: tj.make_beams(pl, [LAUNCHER, LAUNCHER], 0.5, PSI, options=_opts(), ctx=CTX,
                                                   device_launch=True, exact_sum=exact),
        "make_beam_series": lambda: tj.make_beam_series([a, b], *beam, options=_opts(), ctx=CTX, exact_sum=exact),
    }
    for what, call in calls.items():
        rec.calls.clear()
        try:
            call()
        except AssertionError:
            pass  # a recorder returns no rays; only the calls made up to the trace matter
        assert rec.modes("torj_ctx_set_exact_sum") == [(int(exact), True)], what
        i = rec.names().index("torj_ctx_set_exact_sum")
        assert rec.calls[i][1][0] is CTX, what


def _no_device_multi():
    mg = tj.MultiGPU.__new__(tj.MultiGPU)
    mg.h, mg.n_devices, mg._plasmas = C.c_void_p(0x99), 0, {}
    mg.config = dict(sharding="contiguous", block_rays=1, deterministic=False)
    return mg


@pytest.mark.parametrize("exact", [True, False])
def test_multi_entry_points_set_the_mode_and_keep_the_config(rec, exact):
    mg = _no_device_multi()
    a, b = _plasmas(2)
    pos, dirs = np.tile([2.5, 0.0, 0.4], (4, 1)), np.tile(tj.pol_tor_angles_2_vector(0.5, 0.0), (4, 1))
    mg.trace_bundle(a, pos, dirs, np.full(4, 0.25), 95e9, 1, 0.5, PSI, options=_opts(), exact_sum=exact)
    assert rec.modes("torj_multi_set_exact_sum") == [(int(exact), True)]
    assert rec.calls[rec.names().index("torj_multi_set_exact_sum")][1][0] is mg.h
    rec.calls.clear()
    mg.make_beam_series([a, b], 2.5, 0.0, 0.4, 0.0, 0.5, 0.02, 0.25, 95e9, 1, 0.5, PSI, options=_opts(), exact_sum=exact)
    assert rec.modes("torj_multi_set_exact_sum") == [(int(exact), True)]
    assert "torj_ctx_set_exact_sum" not in rec.names()
    assert mg.config == dict(sharding="contiguous", block_rays=1, deterministic=False)
    mg.h = None  # nothing to destroy


def test_device_less_multi_config_keys():
    mg = _no_device_multi()
    assert set(mg.config) == {"sharding", "block_rays", "deterministic"}
    mg.h = None
