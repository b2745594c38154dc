"""rthx — B200-native Monte Carlo exchange-factor ray tracer behind RayTraceHeatTransfer.jl's
`mesh(N_rays; method=:exchange, rec)` interface.

Host side (this package, Python because Julia is absent from the image) mirrors the reference's operator
interface; the compute path is the hand-written sm_100a CUDA library in csrc/ reached through the C ABI of
include/rthx.h.  There is no CPU fallback: tracing raises if the CUDA library or a B200 is missing.
"""
from .domain import (PolyVolume2D, RayTracingDomain2D, RayRecorder, collect_rays, meshQuad, meshTriangle)
from .flatten import flatten_domain, FlatMesh
from ._lib import (make_trace_args, load_library, library_path, build_library, DeviceTracer, RthxError)
from .tracing import (parallelRayTracing, exchangeRayTracing, computeExchangeFactorsBin, group_uniform_bins,
                      counts_to_F, get_w, get_b)
from .equilibrium import solveEquilibrium, equilibriumGrey2D, buildSystemMatrix
from .direct import directRayTracing
from . import meshes, smoothing

__all__ = [
    "PolyVolume2D", "RayTracingDomain2D", "RayRecorder", "collect_rays", "meshQuad", "meshTriangle",
    "flatten_domain", "FlatMesh", "make_trace_args", "load_library", "library_path", "build_library",
    "DeviceTracer", "RthxError", "parallelRayTracing", "exchangeRayTracing", "computeExchangeFactorsBin",
    "group_uniform_bins", "counts_to_F", "get_w", "get_b", "meshes",
    "solveEquilibrium", "equilibriumGrey2D", "buildSystemMatrix", "directRayTracing",
]
