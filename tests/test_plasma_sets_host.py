"""Plasma sets, host side: the argument checks of trace_bundle / marshal_bundle / make_beams that raise before any device
call, and the slice selection of imas.plasmas_from_dd. Runs without a GPU."""
import numpy as np
import pytest

import torj_jl_b200 as tj
from torj_jl_b200 import imas
from torj_jl_b200.solve import marshal_bundle


def _rays(n):
    pos = np.tile([2.5, 0.0, 0.4], (n, 1))
    dirs = np.tile(tj.pol_tor_angles_2_vector(0.5, 0.0), (n, 1))
    return pos, dirs, np.full(n, 1.0 / n)


def test_marshal_checks_beam_plasma():
    pos, dirs, w = _rays(6)
    bid = np.repeat([0, 1, 2], 2)
    psi = np.linspace(0, 1, 10)
    m = marshal_bundle(pos, dirs, w, 95e9, 1, psi, bid, 3, n_plasmas=2, beam_plasma=[0, 1, 1])
    assert m["beam_plasma"].dtype == np.int32 and list(m["beam_plasma"]) == [0, 1, 1]
    assert marshal_bundle(pos, dirs, w, 95e9, 1, psi, bid, 3)["beam_plasma"] is None
    with pytest.raises(ValueError, match="one entry per beam"):
        marshal_bundle(pos, dirs, w, 95e9, 1, psi, bid, 3, n_plasmas=2, beam_plasma=[0, 1])
    with pytest.raises(ValueError, match=r"\[0, 2\)"):
        marshal_bundle(pos, dirs, w, 95e9, 1, psi, bid, 3, n_plasmas=2, beam_plasma=[0, 1, 2])
    with pytest.raises(ValueError, match=r"\[0, 2\)"):
        marshal_bundle(pos, dirs, w, 95e9, 1, psi, bid, 3, n_plasmas=2, beam_plasma=[0, -1, 1])
    with pytest.raises(ValueError, match="several beams"):
        marshal_bundle(pos, dirs, w, 95e9, 1, psi, None, 1, n_plasmas=2, beam_plasma=[1])


def test_trace_bundle_checks_before_the_library():
    arr = tj.solovev_arrays(17, 17)
    pl = tj.Plasma(*arr.values())
    pos, dirs, w = _rays(4)
    psi = np.linspace(0, 1, 10)
    bid = np.array([0, 0, 1, 1])
    with pytest.raises(ValueError, match="needs a sequence"):
        tj.trace_bundle(pl, pos, dirs, w, 95e9, 1, 0.5, psi, beam_id=bid, n_beams=2, beam_plasma=[0, 0])
    with pytest.raises(ValueError, match="needs beam_plasma"):
        tj.trace_bundle([pl, pl], pos, dirs, w, 95e9, 1, 0.5, psi, beam_id=bid, n_beams=2)
    with pytest.raises(ValueError, match=r"\[0, 2\)"):
        tj.trace_bundle([pl, pl], pos, dirs, w, 95e9, 1, 0.5, psi, beam_id=bid, n_beams=2, beam_plasma=[0, 5])
    with pytest.raises(TypeError):
        tj.trace_bundle([], pos, dirs, w, 95e9, 1, 0.5, psi, beam_id=bid, n_beams=2, beam_plasma=[0, 0])
    launchers = [dict(r=2.5, phi=0.0, z=0.4, steering_angle_tor=0.0, steering_angle_pol=0.5, spot_size=0.02,
                      inverse_curvature_radius=0.25, f=95e9, mode=1, plasma=1)]
    with pytest.raises(ValueError, match="single Plasma"):
        tj.make_beams(pl, launchers, 0.5, psi)
    with pytest.raises(ValueError, match=r"\[0, 1\)"):
        tj.make_beams([pl], launchers, 0.5, psi)
    with pytest.raises(ValueError, match="several launchers"):
        tj.make_beams([pl, pl], launchers, 0.5, psi, device_launch=True)


def test_plasmas_from_dd_slice_selection():
    arr = tj.solovev_arrays(17, 19)
    dd = imas.solovev_dd(arr, times=(1.0, 2.0, 3.0), ne_scale_per_slice=(1.0, 2.0, 3.0))
    every = imas.plasmas_from_dd(dd)
    assert len(every) == 3
    for p, t in zip(every, (1.0, 2.0, 3.0)):
        one = imas.plasma_from_dd(dd, t)
        for k in one.coefs:
            assert np.array_equal(p.coefs[k], one.coefs[k]), (t, k)
    picked = imas.plasmas_from_dd(dd, times=[2.5, 1.0, 9.0])  # causal lookup: the slices of t = 2, 1, 3
    for p, t in zip(picked, (2.0, 1.0, 3.0)):
        assert np.array_equal(p.coefs["lnne"], imas.plasma_from_dd(dd, t).coefs["lnne"])
    assert not np.array_equal(picked[0].coefs["lnne"], picked[1].coefs["lnne"])
    with pytest.raises(ValueError):
        imas.plasmas_from_dd(dd, times=[0.5])


def test_plasmas_from_dd_refuses_different_grids():
    dd = imas.solovev_dd(tj.solovev_arrays(17, 17), times=(1.0, 2.0))
    other = imas.solovev_dd(tj.solovev_arrays(17, 17, R_range=(0.5, 2.8)), times=(2.0,))
    dd["equilibrium"]["time_slice"][1] = other["equilibrium"]["time_slice"][0]
    with pytest.raises(ValueError, match="grid"):
        imas.plasmas_from_dd(dd)
    assert len(imas.plasmas_from_dd(dd, times=[1.0, 1.5])) == 2  # both valid at the first slice
