"""Plasma sets on several GPUs, host side: MultiGPU.trace_bundle and MultiGPU.make_beam_series refuse malformed sets
before any library call. The MultiGPU object is built without a device and the library is replaced by one that fails
the test when it is called. Runs without a GPU."""
import numpy as np
import pytest

import torj_jl_b200 as tj
from torj_jl_b200 import _lib


@pytest.fixture
def no_device_multi(monkeypatch):
    arr = tj.solovev_arrays(17, 17)
    pls = [tj.Plasma(*arr.values(), build="device") for _ in range(2)]  # host prefilters only: no device involved

    def no_library():
        raise AssertionError("the library was called before the refusal")

    monkeypatch.setattr(_lib, "lib", no_library)
    mg = tj.MultiGPU.__new__(tj.MultiGPU)
    mg.h, mg.n_devices, mg._plasmas = None, 0, {}
    mg.config = dict(sharding="contiguous", block_rays=1, deterministic=False)
    return mg, pls


def _rays(n):
    pos = np.tile([2.5, 0.0, 0.4], (n, 1))
    dirs = np.tile(tj.pol_tor_angles_2_vector(0.5, 0.0), (n, 1))
    return pos, dirs, np.full(n, 1.0 / n)


def test_multi_trace_bundle_refuses_bad_sets_before_the_library(no_device_multi):
    mg, (a, b) = no_device_multi
    pos, dirs, w = _rays(6)
    psi = np.linspace(0, 1, 10)
    bid = np.repeat([0, 1, 2], 2)
    with pytest.raises(ValueError, match="needs beam_plasma"):
        mg.trace_bundle([a, b], pos, dirs, w, 95e9, 1, 0.5, psi, beam_id=bid, n_beams=3)
    with pytest.raises(ValueError, match="needs a sequence"):
        mg.trace_bundle(a, pos, dirs, w, 95e9, 1, 0.5, psi, beam_id=bid, n_beams=3, beam_plasma=[0, 0, 0])
    for bad in ([0, 1, 2], [0, -1, 1]):
        with pytest.raises(ValueError, match=r"\[0, 2\)"):
            mg.trace_bundle([a, b], pos, dirs, w, 95e9, 1, 0.5, psi, beam_id=bid, n_beams=3, beam_plasma=bad)
    with pytest.raises(ValueError, match="one entry per beam"):
        mg.trace_bundle([a, b], pos, dirs, w, 95e9, 1, 0.5, psi, beam_id=bid, n_beams=3, beam_plasma=[0, 1])
    with pytest.raises(ValueError, match="several beams"):
        mg.trace_bundle([a, b], pos, dirs, w, 95e9, 1, 0.5, psi, beam_plasma=[1])
    with pytest.raises(TypeError):
        mg.trace_bundle([], pos, dirs, w, 95e9, 1, 0.5, psi, beam_id=bid, n_beams=3, beam_plasma=[0, 0, 0])
    assert mg._plasmas == {}  # no per-device copy was made


def test_multi_make_beam_series_refuses_bad_sets_before_the_library(no_device_multi):
    mg, (a, b) = no_device_multi
    psi = np.linspace(0, 1, 10)
    args = (2.5, 0.0, 0.4, 0.0, 0.5, 0.02, 0.25, 95e9, 1, 0.5, psi)
    with pytest.raises(TypeError):
        mg.make_beam_series([], *args)
    with pytest.raises(TypeError):
        mg.make_beam_series([a, "not a plasma"], *args)
    assert mg.config == dict(sharding="contiguous", block_rays=1, deterministic=False) and mg._plasmas == {}
