"""ctypes loader for tests/native/direct_fields_oracle.c — TEST INFRASTRUCTURE: method=:direct with the redirection tally on the CPU,
on the CPU oracle's traversal and Philox stream.  The library is compiled once per process into a temporary directory (the tree may be
read-only)."""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

import rthx
from rthx._abi import rthx_mesh, rthx_trace_args, c_i32p, c_u64p

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_LIB = None


def lib():
    global _LIB
    if _LIB is None:
        so = os.path.join(tempfile.mkdtemp(prefix="rthx_direct_fields_oracle_"), "libdirect_fields_oracle.so")
        cc = "/usr/bin/gcc" if os.access("/usr/bin/gcc", os.X_OK) else (shutil.which("gcc") or "cc")   # the oracle's Makefile pins it too
        subprocess.run([cc, "-O2", "-fPIC", "-fopenmp", "-ffp-contract=off", "-fno-fast-math", "-shared", "-I", os.path.join(ROOT, "include"),
                        "-o", so, os.path.join(ROOT, "tests", "native", "direct_fields_oracle.c"), "-lm"], check=True, capture_output=True)
        L = C.CDLL(so)
        L.rthx_oracle_trace_direct_fields.restype = C.c_int
        L.rthx_oracle_trace_direct_fields.argtypes = [C.POINTER(rthx_mesh), C.POINTER(rthx_trace_args), c_i32p, C.POINTER(C.c_int64), C.c_int32,
                                                      C.POINTER(C.c_uint8), c_u64p, c_u64p, c_u64p, c_u64p, C.c_int]
        _LIB = L
    return _LIB


def trace_direct_fields(flat, sources, rays, reemit, seed=0x5EED0001, band=0, nudge=None, n_threads=0, ray_id_offset=0, specular=False):
    """rthx_trace_direct_fields on the CPU: counts [R, N] u64 and lost [N] u64 as direct_oracle.trace_direct, plus redirected [R, N] u64
    (row y = element sources[y], every scattering or reflection of its bundles at element k in column k) and segments, the traversal
    segments of all bundles."""
    args, keep = rthx.make_trace_args(0, seed=seed, bins=(band,), nudge=nudge, ray_id_offset=ray_id_offset, mode=2 if specular else 1)
    src = np.ascontiguousarray(sources, dtype=np.int32).ravel()
    nr = np.ascontiguousarray(rays, dtype=np.int64).ravel()
    re_ = np.ascontiguousarray(reemit, dtype=np.uint8).ravel()
    N = flat.n_elements
    assert len(nr) == len(src) and len(re_) == N
    counts = np.zeros((len(src), N), np.uint64)
    redirected = np.zeros((len(src), N), np.uint64)
    lost = np.zeros(N, np.uint64)
    segments = C.c_uint64(0)
    rc = lib().rthx_oracle_trace_direct_fields(C.byref(flat.c), C.byref(args), src.ctypes.data_as(c_i32p), nr.ctypes.data_as(C.POINTER(C.c_int64)),
                                               len(src), re_.ctypes.data_as(C.POINTER(C.c_uint8)), counts.ctypes.data_as(c_u64p),
                                               redirected.ctypes.data_as(c_u64p), lost.ctypes.data_as(c_u64p), C.byref(segments), int(n_threads))
    if rc != 0:
        raise RuntimeError(f"rthx_oracle_trace_direct_fields failed with status {rc}")
    return dict(counts=counts, redirected=redirected, lost=lost, segments=int(segments.value))
