"""The Python front ends' library calls, pinned: every public entry point makes the calls of tests/golden/frontend_calls.json,
in that order, with the same scalar arguments, the same NULL / non-NULL pointers, the same option fields and the same
plasma handles, raises the same refusals before any call, and returns results of the same keys, dtypes, shapes and
host-computed values. The library is replaced by a recorder, so this runs without a GPU.

Regenerate the golden log (only when a front end is meant to call the library differently):
    python tests/test_frontend_calls.py"""
import ctypes as C
import hashlib
import json
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torj_jl_b200 as tj  # noqa: E402
from torj_jl_b200 import _lib, solve  # noqa: E402
from torj_jl_b200.distributed import trace_sharded  # noqa: E402

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "frontend_calls.json")
CTX = C.c_void_p(0x1234)
PSI = np.linspace(0.0, 1.0, 12)
N_OUT = 10  # what the recorder writes into an int64 out-argument (rays of a launcher bundle, exact words)
# called from __del__ of Plasma and MultiGPU, whenever the garbage collector gets to them: not part of a call's sequence
FINALIZERS = {"torj_plasma_destroy", "torj_multi_plasma_destroy", "torj_multi_destroy"}


class CallLog:
    """Stands in for libtorj_cuda.so: every function returns 0 and is logged. A handle out-argument gets a distinct
    value; pointers are logged as NULL (None) or non-NULL, by-reference structs by their fields, plasma arrays by their
    handles."""

    def __init__(self):
        self.calls = []
        self.next_handle = 0x1000

    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)

        def fn(*args):
            if name not in FINALIZERS:
                self.calls.append([name] + [self.arg(a) for a in args])
            return 0
        return fn

    def arg(self, a):
        if a is None or isinstance(a, (bool, int, float)):
            return a
        if isinstance(a, C.c_void_p):
            return ["handle", a.value]
        if type(a).__name__ == "CArgObject":  # C.byref(x)
            x = a._obj
            if isinstance(x, C.Structure):
                return [type(x).__name__] + [getattr(x, k) for k, _ in x._fields_]
            if isinstance(x, C.c_void_p):
                self.next_handle += 0x10
                x.value = self.next_handle
                return ["out handle", x.value]
            if isinstance(x, C.c_int64):
                x.value = N_OUT
                return "out int64"
            raise TypeError(f"unexpected by-reference argument {x!r}")
        if isinstance(a, C.Array):
            return ["plasmas", list(a)]
        if isinstance(a, C._Pointer):
            return "ptr" if a else "NULL"
        raise TypeError(f"unexpected argument {a!r}")


def describe(v):
    """A result's structure and host-side values: arrays by dtype, shape and a hash of their bytes."""
    if isinstance(v, dict):
        return {str(k): describe(x) for k, x in v.items()}
    if isinstance(v, (list, tuple)):
        return [describe(x) for x in v]
    if isinstance(v, np.ndarray):
        return ["ndarray", str(v.dtype), list(v.shape), hashlib.sha256(np.ascontiguousarray(v).tobytes()).hexdigest()[:16]]
    if isinstance(v, (bool, int, float, str)) or v is None:
        return [type(v).__name__, v]
    return [type(v).__name__]


def _opts():
    o = _lib.TorjOptions()
    o.n_segments, o.dtmax = 100, 1e-4
    return o


def _plasmas(k):
    arr = tj.solovev_arrays(17, 17)
    return [tj.Plasma(*arr.values(), build="device") for _ in range(k)]  # host prefilters only: no device involved


def _bundle(n=4):
    return np.tile([2.5, 0.0, 0.4], (n, 1)), np.tile(tj.pol_tor_angles_2_vector(0.5, 0.0), (n, 1)), np.full(n, 0.25)


def _multi():
    mg = tj.MultiGPU.__new__(tj.MultiGPU)
    mg.h, mg.n_devices, mg._plasmas = C.c_void_p(0x99), 0, {}
    mg.config = dict(sharding="contiguous", block_rays=1, deterministic=False)
    return mg


BEAM = (2.5, 0.1, 0.4, 0.05, 0.5, 0.02, 0.25, 95e9, 1, 0.5, PSI)


def _launchers(plasma_keys=False):
    out = []
    for b in range(3):
        q = dict(r=2.5 - 0.1 * b, phi=0.3 * b, z=0.4 + 0.05 * b, steering_angle_tor=0.02 * b, steering_angle_pol=0.5 + 0.1 * b,
                 spot_size=0.02 + 0.001 * b, inverse_curvature_radius=0.25, f=95e9 + 1e9 * b, mode=1 + b % 2)
        if plasma_keys:
            q["plasma"] = b % 2
        out.append(q)
    return out


def _trace_bundle(case):
    pos, dirs, w = _bundle()
    kw = dict(options=_opts(), ctx=CTX)
    if case in ("set", "set exact", "set reduce_exact"):
        a, b = _plasmas(2)
        pl = [a, b]
        kw.update(beam_id=[0, 0, 1, 1], n_beams=2, beam_plasma=[1, 0])
    else:
        pl, = _plasmas(1)
    if case == "window":
        kw.update(trajectories=(1, 2))
    if case == "window max_pts":
        kw.update(trajectories=(0, 3), traj_max_pts=40)
    if "exact" in case:
        kw.update(exact_sum=True)
    if "reduce_exact" in case:
        kw.update(reduce_exact=lambda words: None)
    if case == "reduce_exact window":
        kw.update(trajectories=(2, 2))
    return tj.trace_bundle(pl, pos, dirs, w, 95e9, 1, 0.5, PSI, **kw)


def _sharded(exact, multibeam):
    pos, dirs, w = _bundle(6)
    w = w * np.arange(1.0, 7.0)
    xs = dict(exact_sum=True) if exact else {}
    if multibeam:
        a, b = _plasmas(2)

        def fn(p, d, wt, beam_id, **k):
            return tj.trace_bundle([a, b], p, d, wt, 95e9, 1, 0.5, PSI, options=_opts(), ctx=CTX, beam_id=beam_id, n_beams=2,
                                   beam_plasma=[0, 1], **xs, **k)
        return trace_sharded(fn, pos, dirs, w, n_beams=2, per_ray={"beam_id": np.array([0, 0, 0, 1, 1, 1])}, **xs)
    pl, = _plasmas(1)

    def fn(p, d, wt, **k):
        return tj.trace_bundle(pl, p, d, wt, 95e9, 1, 0.5, PSI, options=_opts(), ctx=CTX, **xs, **k)
    return trace_sharded(fn, pos, dirs, w, **xs)


def _series(multi):
    a, b, c = _plasmas(3)
    if multi:
        return _multi().make_beam_series([a, b, c], *BEAM, options=_opts(), exact_sum=True)
    return tj.make_beam_series([a, b, c], *BEAM, options=_opts(), ctx=CTX, exact_sum=True)


def _multi_trace(case):
    pos, dirs, w = _bundle()
    if case == "set":
        a, b = _plasmas(2)
        return _multi().trace_bundle([a, b], pos, dirs, w, np.full(4, 95e9), np.ones(4, dtype=np.int32), 0.5, PSI,
                                     options=_opts(), beam_id=[0, 0, 1, 1], n_beams=2, beam_plasma=[1, 0])
    pl, = _plasmas(1)
    return _multi().trace_bundle(pl, pos, dirs, w, 95e9, 1, 0.5, PSI, options=_opts(), exact_sum=True)


def _refusal(case):
    pos, dirs, w = _bundle()
    pl, = _plasmas(1)
    a, b = _plasmas(2)
    kw = dict(options=_opts(), ctx=CTX)
    if case == "reduce_exact without exact_sum":
        return tj.trace_bundle(pl, pos, dirs, w, 95e9, 1, 0.5, PSI, reduce_exact=lambda words: None, **kw)
    if case == "beam_plasma without a set":
        return tj.trace_bundle(pl, pos, dirs, w, 95e9, 1, 0.5, PSI, beam_plasma=[0], **kw)
    if case == "set without beam_plasma":
        return tj.trace_bundle([a, b], pos, dirs, w, 95e9, 1, 0.5, PSI, **kw)
    if case == "not a plasma":
        return tj.trace_bundle([a, "b"], pos, dirs, w, 95e9, 1, 0.5, PSI, beam_plasma=[0], **kw)
    if case == "beam_plasma out of range":
        return tj.trace_bundle([a, b], pos, dirs, w, 95e9, 1, 0.5, PSI, beam_id=[0, 0, 1, 1], n_beams=2, beam_plasma=[0, 2],
                               **kw)
    if case == "set with one beam":
        return tj.trace_bundle([a, b], pos, dirs, w, 95e9, 1, 0.5, PSI, beam_plasma=[1], **kw)
    if case == "beam_id length":
        return tj.trace_bundle(pl, pos, dirs, w, 95e9, 1, 0.5, PSI, beam_id=[0, 1], n_beams=2, **kw)
    if case == "multi set without beam_plasma":
        return _multi().trace_bundle([a, b], pos, dirs, w, 95e9, 1, 0.5, PSI, options=_opts())
    if case == "launcher plasma on one plasma":
        return tj.make_beams(pl, _launchers(True), 0.5, PSI, **kw)
    if case == "launcher plasma out of range":
        return tj.make_beams([a], _launchers(True), 0.5, PSI, device_launch=True, **kw)
    if case == "device launch N_rings":
        return tj.make_beams(pl, _launchers(), 0.5, PSI, device_launch=True, N_rings=1, **kw)
    if case == "device launch set with one launcher":
        return tj.make_beams([a, b], _launchers(True)[1:2], 0.5, PSI, device_launch=True, **kw)
    if case == "sharded exact without rays":
        return trace_sharded(lambda *x, **k: None, np.zeros((0, 3)), np.zeros((0, 3)), np.zeros(0), exact_sum=True)
    raise KeyError(case)


CASES = {
    "trace_bundle plasma": lambda: _trace_bundle("plasma"),
    "trace_bundle set": lambda: _trace_bundle("set"),
    "trace_bundle window": lambda: _trace_bundle("window"),
    "trace_bundle window max_pts": lambda: _trace_bundle("window max_pts"),
    "trace_bundle exact": lambda: _trace_bundle("exact"),
    "trace_bundle set exact": lambda: _trace_bundle("set exact"),
    "trace_bundle reduce_exact": lambda: _trace_bundle("reduce_exact"),
    "trace_bundle reduce_exact window": lambda: _trace_bundle("reduce_exact window"),
    "trace_bundle set reduce_exact": lambda: _trace_bundle("set reduce_exact"),
    "make_ray": lambda: tj.make_ray(_plasmas(1)[0], [2.5, 0.0, 0.4], tj.pol_tor_angles_2_vector(0.5, 0.0), 95e9, 1, 0.5, PSI,
                                    options=_opts(), ctx=CTX),
    "make_beam": lambda: tj.make_beam(_plasmas(1)[0], *BEAM, options=_opts(), ctx=CTX, exact_sum=True),
    "make_beams host": lambda: tj.make_beams(_plasmas(1)[0], _launchers(), 0.5, PSI, options=_opts(), ctx=CTX),
    "make_beams host set": lambda: tj.make_beams(_plasmas(2), _launchers(True), 0.5, PSI, options=_opts(), ctx=CTX,
                                                 exact_sum=True, N_rings=2),
    "make_beams device": lambda: tj.make_beams(_plasmas(1)[0], _launchers(), 0.5, PSI, options=_opts(), ctx=CTX,
                                               device_launch=True, exact_sum=True),
    "make_beams host one launcher": lambda: tj.make_beams(_plasmas(1)[0], _launchers()[2:], 0.5, PSI, options=_opts(),
                                                          ctx=CTX),
    "make_beams device one launcher": lambda: tj.make_beams(_plasmas(1)[0], _launchers()[2:], 0.5, PSI, options=_opts(),
                                                            ctx=CTX, device_launch=True),
    "make_beams device set": lambda: tj.make_beams(_plasmas(2), _launchers(True), 0.5, PSI, options=_opts(), ctx=CTX,
                                                   device_launch=True, N_rings=4, min_azimuthal_points=6,
                                                   normalize_weight_sum=False),
    "make_beam_series": lambda: _series(False),
    "MultiGPU.trace_bundle plasma": lambda: _multi_trace("plasma"),
    "MultiGPU.trace_bundle set": lambda: _multi_trace("set"),
    "MultiGPU.make_beam_series": lambda: _series(True),
    "trace_sharded float": lambda: _sharded(False, False),
    "trace_sharded float beams": lambda: _sharded(False, True),
    "trace_sharded exact": lambda: _sharded(True, False),
    "trace_sharded exact beams": lambda: _sharded(True, True),
}
REFUSALS = ["reduce_exact without exact_sum", "beam_plasma without a set", "set without beam_plasma", "not a plasma",
            "beam_plasma out of range", "set with one beam", "beam_id length", "multi set without beam_plasma",
            "launcher plasma on one plasma", "launcher plasma out of range", "device launch N_rings",
            "device launch set with one launcher", "sharded exact without rays"]
for _r in REFUSALS:
    CASES["refusal: " + _r] = (lambda r: lambda: _refusal(r))(_r)


def record(case, monkeypatch):
    """(the calls, the result or the refusal) of one case"""
    log = CallLog()
    monkeypatch.setattr(_lib, "lib", lambda: log)
    # the recorder hands out no device memory: the words and the profile are host tensors of the right length
    monkeypatch.setattr(solve, "device_tensor", lambda ptr, n, typestr: torch.zeros(
        int(n), dtype=torch.int64 if typestr == "<i8" else torch.float64))
    try:
        out = ["result", describe(CASES[case]())]
    except Exception as e:  # a refusal: its type and text
        out = ["raises", type(e).__name__, str(e)]
    return json.loads(json.dumps(dict(calls=log.calls, out=out)))


def _golden():
    with open(GOLDEN) as fh:
        return json.load(fh)


@pytest.mark.parametrize("case", list(CASES))
def test_frontend_calls(case, monkeypatch):
    want = _golden()[case]
    got = record(case, monkeypatch)
    if got["out"][0] == "raises":  # a refusal comes before any library call that is not the plasma's own set-up
        assert not [c for c in got["calls"] if not c[0].startswith(("torj_bspline_prefilter", "torj_multi_configure"))]
    assert got["calls"] == want["calls"]
    assert got["out"] == want["out"]


def test_golden_covers_every_case():
    assert sorted(_golden()) == sorted(CASES)


if __name__ == "__main__":
    mp = pytest.MonkeyPatch()
    log = {}
    for case in CASES:
        with mp.context() as m:
            log[case] = record(case, m)
    with open(GOLDEN, "w") as fh:
        fh.write("{\n" + ",\n".join(
            json.dumps(case) + ': {"calls": [\n' + ",\n".join(json.dumps(c) for c in v["calls"]) + '\n], "out": '
            + json.dumps(v["out"]) + "}" for case, v in log.items()) + "\n}\n")
    print(f"wrote {GOLDEN}: {len(log)} cases, {sum(len(v['calls']) for v in log.values())} calls")
