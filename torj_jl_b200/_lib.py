"""ctypes binding of libtorj_cuda.so (include/torj_cuda.h). There is no CPU fallback: if the CUDA library is
missing, importing this module's `lib()` raises, and so does every entry point without a CUDA device."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("TORJ_CUDA_LIB") or os.path.join(_HERE, "libtorj_cuda.so")  # override: tuning experiments
_LIB = None

c_dp = C.POINTER(C.c_double)
c_ip = C.POINTER(C.c_int32)
c_vp = C.c_void_p


class TorjOptions(C.Structure):
    """torj_options: solver constants the reference hard-codes (src/solve.jl:145,157,174,176; src/absorption.jl:194,199)."""
    _fields_ = [("scheme", C.c_int32), ("n_segments", C.c_int32), ("dtmax", C.c_double), ("abstol", C.c_double),
                ("reltol", C.c_double), ("psi_stop", C.c_double), ("p_stop", C.c_double), ("te_min", C.c_double),
                ("max_harmonic", C.c_int32), ("max_steps_per_segment", C.c_int32), ("alpha_floor", C.c_double),
                ("schedule", C.c_int32), ("absorption_model", C.c_int32), ("lanes_per_ray", C.c_int32), ("reserved_", C.c_int32)]


class TorjCounters(C.Structure):
    _fields_ = [("n_acc", C.c_int64), ("n_rej", C.c_int64), ("n_rhs", C.c_int64), ("n_alpha", C.c_int64),
                ("n_harm", C.c_int64), ("n_rays_ok", C.c_int64), ("n_harm_pruned", C.c_int64), ("n_alpha_skipped", C.c_int64)]

    def as_dict(self):
        return {k: int(getattr(self, k)) for k, _ in self._fields_}


class TorjGrid(C.Structure):
    _fields_ = [("nR", C.c_int32), ("nZ", C.c_int32), ("R_first", C.c_double), ("R_last", C.c_double),
                ("Z_first", C.c_double), ("Z_last", C.c_double)]


class TorjError(RuntimeError):
    pass


# every symbol include/torj_cuda.h declares: (restype, argtypes)
SIGNATURES = {
    "torj_options_default": (None, [C.POINTER(TorjOptions)]),
    "torj_last_error": (C.c_char_p, []),
    "torj_abi_version": (C.c_int, []),
    "torj_ctx_create": (C.c_int, [C.c_int, c_vp, C.POINTER(c_vp)]),
    "torj_ctx_destroy": (None, [c_vp]),
    "torj_ctx_sync": (C.c_int, [c_vp]),
    "torj_ctx_launch_count": (C.c_int64, [c_vp]),
    "torj_ctx_last_trace_ms": (C.c_int, [c_vp, c_dp]),
    "torj_ctx_set_exact_sum": (C.c_int, [c_vp, C.c_int32]),
    "torj_abs_init": (C.c_int, [c_vp, C.c_int32, c_dp, c_dp]),
    "torj_warm_alpha": (C.c_int, [c_vp, C.c_int64, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp, C.c_int32, c_dp, c_dp, c_ip, c_ip]),
    "torj_bspline_prefilter_2d": (C.c_int, [C.c_int32, C.c_int32, c_dp, c_dp]),
    "torj_bspline_prefilter_1d": (C.c_int, [C.c_int32, c_dp, c_dp]),
    "torj_plasma_create": (C.c_int, [c_vp, C.POINTER(TorjGrid), c_dp, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp, C.c_int32,
                                     C.c_double, C.c_double, C.c_double, C.POINTER(c_vp)]),
    "torj_plasma_create_from_data": (C.c_int, [c_vp, C.POINTER(TorjGrid), c_dp, c_dp, c_dp, c_dp, C.c_int32, c_dp, c_dp, c_dp,
                                               c_dp, c_dp, C.c_int32, C.POINTER(c_vp)]),
    "torj_plasma_destroy": (None, [c_vp]),
    "torj_probe": (C.c_int, [c_vp, c_vp, C.POINTER(TorjOptions), C.c_int64, c_dp, c_dp, C.c_double, C.c_int32, c_dp]),
    "torj_rhs": (C.c_int, [c_vp, c_vp, C.POINTER(TorjOptions), C.c_int64, c_dp, C.c_double, C.c_int32, c_dp]),
    "torj_bundle_create": (C.c_int, [c_vp, C.c_int64, c_dp, c_dp, c_dp, c_dp, c_ip, C.c_int32, C.POINTER(c_vp)]),
    "torj_bundle_create_from_launchers": (C.c_int, [c_vp, C.c_int32, c_dp, c_dp, c_dp, c_dp, c_dp, c_ip, C.c_int32, C.c_int32,
                                                    C.c_int32, c_dp, c_dp, C.POINTER(c_vp), C.POINTER(C.c_int64)]),
    "torj_bundle_rays": (C.c_int, [c_vp, c_dp, c_dp, c_dp]),
    "torj_bundle_destroy": (None, [c_vp]),
    "torj_bundle_set_window": (C.c_int, [c_vp, C.c_int64, C.c_int64, C.c_int32]),
    "torj_bundle_set_beams": (C.c_int, [c_vp, C.c_int32, c_ip]),
    "torj_bundle_trace": (C.c_int, [c_vp, c_vp, C.POINTER(TorjOptions), C.c_double, C.c_int32, c_dp]),
    "torj_bundle_trace_plasmas": (C.c_int, [c_vp, C.c_int32, C.POINTER(c_vp), c_ip, C.POINTER(TorjOptions), C.c_double,
                                            C.c_int32, c_dp]),
    "torj_bundle_device_profile": (c_vp, [c_vp]),
    "torj_bundle_results": (C.c_int, [c_vp, c_dp, c_dp, c_dp, c_dp, c_ip, c_ip, C.POINTER(TorjCounters)]),
    "torj_bundle_trajectories": (C.c_int, [c_vp, c_dp, c_dp, c_dp, c_dp, c_dp]),
    "torj_bundle_final_state": (C.c_int, [c_vp, c_dp, c_dp, c_dp, c_dp]),
    "torj_bundle_trajectories_cyl": (C.c_int, [c_vp, c_dp, c_dp, c_dp]),
    "torj_trace": (C.c_int, [c_vp, c_vp, C.POINTER(TorjOptions), C.c_int64, c_dp, c_dp, c_dp, c_dp, c_ip, C.c_int32,
                             C.c_double, C.c_int32, c_dp, C.c_int32, c_ip, c_dp, c_dp, c_dp, c_dp, c_ip, c_ip, C.c_int64, C.c_int64,
                             C.c_int32, c_dp, c_dp, c_dp, c_dp, c_dp, C.POINTER(TorjCounters)]),
    "torj_trace_plasmas": (C.c_int, [c_vp, C.c_int32, C.POINTER(c_vp), c_ip, C.POINTER(TorjOptions), C.c_int64, c_dp, c_dp, c_dp,
                                     c_dp, c_ip, C.c_int32, C.c_double, C.c_int32, c_dp, C.c_int32, c_ip, c_dp, c_dp, c_dp, c_dp,
                                     c_ip, c_ip, C.c_int64, C.c_int64, C.c_int32, c_dp, c_dp, c_dp, c_dp, c_dp,
                                     C.POINTER(TorjCounters)]),
    "torj_multi_create": (C.c_int, [C.c_int32, C.POINTER(c_vp)]),
    "torj_multi_destroy": (None, [c_vp]),
    "torj_multi_device_count": (C.c_int32, [c_vp]),
    "torj_multi_configure": (C.c_int, [c_vp, C.c_int32, C.c_int64, C.c_int32]),
    "torj_multi_used_nccl": (C.c_int32, [c_vp]),
    "torj_multi_abs_init": (C.c_int, [c_vp, C.c_int32, c_dp, c_dp]),
    "torj_multi_set_exact_sum": (C.c_int, [c_vp, C.c_int32]),
    "torj_multi_last_trace_ms": (C.c_int, [c_vp, C.c_int32, c_dp]),
    "torj_multi_plasma_create_from_data": (C.c_int, [c_vp, C.POINTER(TorjGrid), c_dp, c_dp, c_dp, c_dp, C.c_int32, c_dp, c_dp,
                                                     c_dp, c_dp, c_dp, C.c_int32, C.POINTER(c_vp)]),
    "torj_multi_plasma_destroy": (None, [c_vp]),
    "torj_multi_trace": (C.c_int, [c_vp, c_vp, C.POINTER(TorjOptions), C.c_int64, c_dp, c_dp, c_dp, c_dp, c_ip, C.c_int32,
                                   C.c_double, C.c_int32, c_dp, C.c_int32, c_ip, c_dp, c_dp, c_dp, c_dp, c_ip, c_ip, C.c_int64,
                                   C.c_int64, C.c_int32, c_dp, c_dp, c_dp, c_dp, c_dp, C.POINTER(TorjCounters)]),
    "torj_multi_trace_plasmas": (C.c_int, [c_vp, C.c_int32, C.POINTER(c_vp), c_ip, C.POINTER(TorjOptions), C.c_int64, c_dp, c_dp,
                                           c_dp, c_dp, c_ip, C.c_int32, C.c_double, C.c_int32, c_dp, C.c_int32, c_ip, c_dp, c_dp,
                                           c_dp, c_dp, c_ip, c_ip, C.c_int64, C.c_int64, C.c_int32, c_dp, c_dp, c_dp, c_dp, c_dp,
                                           C.POINTER(TorjCounters)]),
    "torj_fp64_peak": (C.c_int, [c_vp, C.c_int32, c_dp, c_dp]),
    "torj_fp64_latency": (C.c_int, [c_vp, C.c_int32, c_dp]),
    "torj_math_probe": (C.c_int, [c_vp, C.c_int64, c_dp, c_dp]),
}


def lib():
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise TorjError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                            "(make -C torj_jl_b200/csrc). torj_jl_b200 has no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _LIB = L
    return _LIB


def check(rc: int):
    if rc != 0:
        raise TorjError(lib().torj_last_error().decode("utf-8", "replace"))


def default_options(**kw) -> TorjOptions:
    o = TorjOptions()
    lib().torj_options_default(C.byref(o))
    for k, v in kw.items():
        if not hasattr(o, k):
            raise AttributeError(f"torj_options has no field {k!r}")
        setattr(o, k, v)
    return o


_CTX = {}


def context(device: int | None = None, stream: int | None = None):
    """Process-wide context per device (device defaults to LOCAL_RANK, else 0)."""
    if device is None:
        device = int(os.environ.get("LOCAL_RANK", "0"))
    key = (device, stream)
    if key not in _CTX:
        h = c_vp()
        check(lib().torj_ctx_create(device, c_vp(stream) if stream else None, C.byref(h)))
        _CTX[key] = h
    return _CTX[key]
