"""ort_b200 -- host side of the B200-native batched sequential ray tracer.

Mirrors the public API of Sagnac/OpticalRayTracing.jl for its data-parallel hot path (solve,
raytrace, full_trace, transfer, reverse_transfer, wavegrad, TSA ...) on top of the C ABI of
libort_b200.so (include/ort_b200.h).  The Julia shim a maintainer would add is in
julia/OpticalRayTracingB200.jl; Julia is not installed in this environment, so this Python
mirror is what drives the same ABI in tests and benchmarks.
"""
from . import _lib, distributed, host, prescriptions
from ._lib import (EXT_OPD, EXT_VIGNETTE, FAST, STRICT, FLAG_CLIP, FLAG_DOMAIN, FLAG_MISS, FLAG_TIR, FLAG_VIGN,
                   Context, OrtError, PinnedArray, STATS_BYTES, STATS_DTYPE)
from .host import (LAMBDA, SA, TSA, Aberration, aberrations, seidel_merit, Wavefront, aim_rays, wavefront, Layout, Lens, RayBasis, RealRay, RealRayError, System,
                   VectorRealRay, flatten, full_trace, full_trace_candidates, full_trace_fields, make_lens, merge_stats,
                   raytrace, reverse_transfer, rms_from_stats, set_default_backend, solve, through_focus, ThroughFocus,
                   trace_chief_ray, trace_edge_rays, trace_marginal_ray, transfer, transfer_matrix,
                   vignetting, Vignetting, wavegrad)

__all__ = ["_lib", "distributed", "host", "prescriptions", "Context", "OrtError", "PinnedArray", "STATS_DTYPE", "FAST",
           "STRICT", "FLAG_MISS", "FLAG_TIR", "FLAG_DOMAIN", "FLAG_CLIP", "FLAG_VIGN", "EXT_OPD", "EXT_VIGNETTE", "STATS_BYTES", "LAMBDA", "SA", "TSA", "Aberration", "aberrations", "seidel_merit", "Wavefront", "aim_rays", "wavefront",
           "Layout", "Lens", "RayBasis", "RealRay", "RealRayError", "System", "VectorRealRay",
           "flatten", "full_trace", "full_trace_candidates", "full_trace_fields", "make_lens", "merge_stats", "raytrace",
           "reverse_transfer", "rms_from_stats", "set_default_backend", "solve", "through_focus", "ThroughFocus", "trace_chief_ray",
           "trace_edge_rays", "trace_marginal_ray", "transfer", "transfer_matrix", "vignetting", "Vignetting", "wavegrad"]
