"""torj_jl_b200 — B200-native ray-tracing hot path of TorJ.jl behind TorJ's own entry points.

Host side (this package, Python because Julia is not installed here) mirrors the reference's names and argument
meaning: Plasma, launch_peripheral_rays, abs_Al_init, make_ray, make_beam.  All numerics of the path run in
libtorj_cuda.so (hand-written sm_100a CUDA, C ABI in include/torj_cuda.h); there is no CPU fallback."""
from ._lib import TorjError, TorjOptions, context, default_options, lib  # noqa: F401
from .absorption import abs_Al_init, alpha_approx, warm_alpha  # noqa: F401
from .launch import launch_peripheral_rays  # noqa: F401
from .multi import MultiGPU  # noqa: F401
from .plasma import Plasma, evaluate_psi  # noqa: F401
from .solve import cylindrical_state, make_beam, make_beam_series, make_beams, make_ray, trace_bundle  # noqa: F401
from .synthetic import pol_tor_angles_2_vector, solovev_arrays  # noqa: F401
from .imas import plasma_arrays_from_dd, plasma_from_dd, plasma_from_imas_json, plasmas_from_dd, solovev_dd  # noqa: F401
