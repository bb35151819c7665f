"""trace_bundle(..., exact_sum=True, reduce_exact=fn), host side: the two C symbols of the exact words and their bindings
exist, reduce_exact without exact_sum is refused before any library call, and the resident-bundle route makes its calls
in the order the cross-process sum needs: trace, words, fn, conversion, results, destroy (also when fn raises).
The library is replaced by the recorder of test_exact_sum_host.py, so this runs without a GPU."""
import ctypes as C
import inspect

import numpy as np
import pytest
import torch

import torj_jl_b200 as tj
from torj_jl_b200 import _lib, solve
from torj_jl_b200.distributed import trace_sharded

from test_exact_sum_host import CTX, PSI, Recorder, _opts, _plasmas


def test_symbols_and_signatures():
    L = _lib.lib()
    assert hasattr(L, "torj_bundle_device_exact_words") and hasattr(L, "torj_bundle_finalize_exact")
    assert _lib.SIGNATURES["torj_bundle_device_exact_words"] == (C.c_int, [_lib.c_vp, C.POINTER(_lib.c_vp),
                                                                          C.POINTER(C.c_int64)])
    assert _lib.SIGNATURES["torj_bundle_finalize_exact"] == (C.c_int, [_lib.c_vp])
    p = inspect.signature(tj.trace_bundle).parameters["reduce_exact"]
    assert p.kind is inspect.Parameter.KEYWORD_ONLY and p.default is None
    p = inspect.signature(trace_sharded).parameters["exact_sum"]
    assert p.kind is inspect.Parameter.KEYWORD_ONLY and p.default is False


@pytest.fixture
def rec(monkeypatch):
    r = Recorder()
    monkeypatch.setattr(_lib, "lib", lambda: r)
    # the recorder hands out no device memory: the words and the profile are host tensors of the right length
    monkeypatch.setattr(solve, "device_tensor", lambda ptr, n, typestr: torch.zeros(
        int(n), dtype=torch.int64 if typestr == "<i8" else torch.float64))
    return r


def _bundle(n=4):
    return np.tile([2.5, 0.0, 0.4], (n, 1)), np.tile(tj.pol_tor_angles_2_vector(0.5, 0.0), (n, 1)), np.full(n, 0.25)


def test_reduce_exact_needs_exact_sum(rec):
    pl, = _plasmas(1)
    pos, dirs, w = _bundle()
    rec.calls.clear()
    with pytest.raises(ValueError, match="exact_sum=True"):
        tj.trace_bundle(pl, pos, dirs, w, 95e9, 1, 0.5, PSI, options=_opts(), ctx=CTX, reduce_exact=lambda words: None)
    assert rec.calls == []


ORDER = ["torj_ctx_set_exact_sum", "torj_bundle_create", "torj_bundle_set_beams", "torj_bundle_set_window", "trace",
         "torj_bundle_device_exact_words", "hook", "torj_bundle_finalize_exact", "torj_bundle_results", "torj_bundle_destroy"]


def _order(rec):
    keep = set(ORDER) | {"torj_bundle_trace", "torj_bundle_trace_plasmas", "torj_bundle_trajectories"}
    return ["trace" if n in ("torj_bundle_trace", "torj_bundle_trace_plasmas") else n for n in rec.names() if n in keep]


@pytest.mark.parametrize("case", ["one plasma", "plasma set", "window"])
def test_reduce_exact_call_order(rec, case):
    pl, = _plasmas(1)
    a, b = _plasmas(2)
    pos, dirs, w = _bundle()
    seen = []

    def hook(words):
        assert words.dtype == torch.int64
        seen.append(words)
        rec.calls.append(("hook", ()))

    kw = dict(options=_opts(), ctx=CTX, exact_sum=True, reduce_exact=hook)
    if case == "plasma set":
        r = tj.trace_bundle([a, b], pos, dirs, w, 95e9, 1, 0.5, PSI, beam_id=[0, 0, 1, 1], n_beams=2, beam_plasma=[0, 1], **kw)
        assert "torj_bundle_trace_plasmas" in rec.names() and "torj_trace_plasmas" not in rec.names()
        assert r["sum_weights"].shape == (2,) and r["dP_dV"].shape == (2, len(PSI))
        assert r["local_vector"].shape == (2 * (len(PSI) + 2),)
    else:
        r = tj.trace_bundle(pl, pos, dirs, w, 95e9, 1, 0.5, PSI, trajectories=(1, 2) if case == "window" else None, **kw)
        assert isinstance(r["sum_weights"], float) and r["local_vector"].shape == (len(PSI) + 2,)
    assert "torj_trace" not in rec.names()
    want = list(ORDER)
    if case == "window":
        want.insert(want.index("torj_bundle_destroy"), "torj_bundle_trajectories")
    assert _order(rec) == want
    assert len(seen) == 1
    assert rec.calls[rec.names().index("torj_ctx_set_exact_sum")][1] == (CTX, 1)
    # the library's stream is idle before fn reads the words
    names = rec.names()
    i_trace = max(i for i, n in enumerate(names) if n in ("torj_bundle_trace", "torj_bundle_trace_plasmas"))
    assert i_trace < names.index("torj_ctx_sync") < names.index("hook")
    for k in ("dP_dV", "deposited_power", "P_final", "P_deposited_ray", "n_points", "status", "counters", "traj_s", "traj_xyz",
              "traj_P", "traj_dP_ds", "traj_dP_dV_ray"):
        assert k in r, k


def test_bundle_is_destroyed_when_the_hook_raises(rec):
    pl, = _plasmas(1)
    pos, dirs, w = _bundle()

    def hook(words):
        raise KeyError("peer gone")

    with pytest.raises(KeyError, match="peer gone"):
        tj.trace_bundle(pl, pos, dirs, w, 95e9, 1, 0.5, PSI, options=_opts(), ctx=CTX, exact_sum=True, reduce_exact=hook)
    names = rec.names()
    assert names[-1] == "torj_bundle_destroy"
    assert "torj_bundle_finalize_exact" not in names and "torj_bundle_results" not in names


def test_bundle_is_destroyed_when_the_trace_fails(rec, monkeypatch):
    pl, = _plasmas(1)
    pos, dirs, w = _bundle()
    real = rec.__getattr__

    def failing(name):
        if name == "torj_bundle_trace":
            return lambda *a: (rec.calls.append((name, a)), 2)[1]
        if name == "torj_last_error":
            return lambda: b"refused"
        return real(name)
    monkeypatch.setattr(Recorder, "__getattr__", lambda self, name: failing(name))
    hook_calls = []
    with pytest.raises(_lib.TorjError, match="refused"):
        tj.trace_bundle(pl, pos, dirs, w, 95e9, 1, 0.5, PSI, options=_opts(), ctx=CTX, exact_sum=True,
                        reduce_exact=hook_calls.append)
    assert hook_calls == [] and rec.names()[-1] == "torj_bundle_destroy"
