"""ctypes binding of the C ABI in include/rthx.h (the Python twin of the Julia `ccall` shim, julia/RTHXExchange.jl).

The shared library `csrc/librthx.so` is built in-tree by `build_library()` (nvcc, sm_100a).  There is no CPU
fallback: if the library is missing or no device is usable, every compute call raises `RthxError`.
"""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess
from typing import Optional, Sequence

import numpy as np

from ._abi import (rthx_mesh, rthx_trace_args, rthx_rec_out, rthx_stats, rthx_info, rthx_smooth_stats, rthx_sparse_stats, c_i32p, c_f64p, c_u64p,
                   rthx_solve_args, rthx_solve_stats, c_i64p,
                   RTHX_SMOOTH_FROM_LAST_TRACE, RTHX_SMOOTH_FROM_COUNTS, RTHX_SMOOTH_FROM_F, RTHX_SMOOTH_FROM_CSC,
                   RTHX_SOLVE_FROM_LAST_SMOOTH, RTHX_SOLVE_FROM_DENSE, RTHX_SOLVE_FROM_CSC, RTHX_ROW_MAJOR, RTHX_COL_MAJOR,
                   RTHX_FIRST_INTERACTION, RTHX_LOCATOR_AUTO, RTHX_LOCATOR_GENERIC, EXPORTED_SYMBOLS)

_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(_HERE, "csrc")
_LIB = None

DEFAULT_SEED = 0x5EED0001
DEFAULT_NUDGE = 10_000 * float(np.finfo(np.float64).eps)  # multiDispatchRayTrace2D.jl:10


class RthxError(RuntimeError):
    pass


def library_path() -> str:
    # RTHX_LIBRARY: another build of the library, e.g. of an earlier commit for an A/B run against this one; never a fallback
    return os.environ.get("RTHX_LIBRARY") or os.path.join(_CSRC, "librthx.so")


def build_library(force: bool = False, verbose: bool = False) -> str:
    """Compile csrc/*.cu into csrc/librthx.so for sm_100a (nvcc cross-compiles without a GPU)."""
    so = library_path()
    srcs = [os.path.join(_CSRC, f) for f in sorted(os.listdir(_CSRC)) if f.endswith((".cu", ".cuh", ".h"))]
    srcs.append(os.path.join(os.path.dirname(_HERE), "include", "rthx.h"))
    if not force and os.path.exists(so) and all(os.path.getmtime(so) >= os.path.getmtime(s) for s in srcs):
        return so
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
           "-Xcompiler", "-fPIC,-O2", "-shared", "--fmad=true",
           "-I", os.path.join(os.path.dirname(_HERE), "include"), "-I", _CSRC,
           "-o", so] + [s for s in srcs if s.endswith(".cu")]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
    env = dict(os.environ)
    env.pop("CC", None)
    env.pop("CXX", None)
    r = subprocess.run(cmd, capture_output=True, text=True, env=env)
    if r.returncode != 0:
        raise RthxError("nvcc failed:\n" + r.stdout + r.stderr)
    if verbose:
        print(r.stdout + r.stderr)
    return so


def load_library():
    """Load csrc/librthx.so (raises RthxError if it has not been built — no fallback)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    so = library_path()
    if not os.path.exists(so):
        raise RthxError(f"{so} not built; run `python -c 'import __graft_entry__ as g; g.build()'` "
                        "(there is no CPU fallback)")
    L = C.CDLL(so)
    L.rthx_create.restype = C.c_int
    L.rthx_create.argtypes = [C.POINTER(C.c_void_p), C.POINTER(rthx_mesh), C.c_int]
    L.rthx_create_multi.restype = C.c_int
    L.rthx_create_multi.argtypes = [C.POINTER(C.c_void_p), C.POINTER(rthx_mesh), C.POINTER(C.c_int), C.c_int]
    L.rthx_device_count.restype = C.c_int
    L.rthx_device_count.argtypes = [C.POINTER(C.c_int)]
    L.rthx_destroy.restype = C.c_int
    L.rthx_destroy.argtypes = [C.c_void_p]
    L.rthx_get_info.restype = C.c_int
    L.rthx_get_info.argtypes = [C.c_void_p, C.POINTER(rthx_info)]
    L.rthx_trace_exchange.restype = C.c_int
    L.rthx_trace_exchange.argtypes = [C.c_void_p, C.POINTER(rthx_trace_args), c_u64p, c_u64p,
                                      C.POINTER(rthx_rec_out), C.POINTER(rthx_stats)]
    L.rthx_trace_exchange_sparse.restype = C.c_int
    L.rthx_trace_exchange_sparse.argtypes = [C.c_void_p, C.POINTER(rthx_trace_args), c_u64p, C.POINTER(rthx_rec_out), C.POINTER(rthx_stats),
                                             C.POINTER(rthx_sparse_stats)]
    L.rthx_trace_exchange_continue.restype = C.c_int
    L.rthx_trace_exchange_continue.argtypes = [C.c_void_p, C.POINTER(rthx_trace_args), c_u64p, C.POINTER(rthx_rec_out), C.POINTER(rthx_stats),
                                               C.POINTER(rthx_sparse_stats)]
    L.rthx_trace_exchange_rows.restype = C.c_int
    L.rthx_trace_exchange_rows.argtypes = [C.c_void_p, C.POINTER(rthx_trace_args), c_i32p, C.c_int32, c_u64p, c_u64p,
                                           C.POINTER(rthx_rec_out), C.POINTER(rthx_stats)]
    L.rthx_trace_direct.restype = C.c_int
    L.rthx_trace_direct.argtypes = [C.c_void_p, C.POINTER(rthx_trace_args), c_i32p, c_i64p, C.c_int32, C.POINTER(C.c_uint8), c_f64p, c_f64p,
                                    c_u64p, c_i64p, C.POINTER(rthx_stats)]
    L.rthx_trace_direct_fields.restype = C.c_int
    L.rthx_trace_direct_fields.argtypes = [C.c_void_p, C.POINTER(rthx_trace_args), c_i32p, c_i64p, C.c_int32, C.POINTER(C.c_uint8), c_f64p, c_f64p,
                                           c_f64p, c_u64p, c_i64p, C.POINTER(rthx_stats)]
    L.rthx_trace_direct_sparse.restype = C.c_int
    L.rthx_trace_direct_sparse.argtypes = [C.c_void_p, C.POINTER(rthx_trace_args), c_i32p, c_i64p, C.c_int32, C.POINTER(C.c_uint8), c_f64p, c_f64p,
                                           c_f64p, c_u64p, c_i64p, C.POINTER(rthx_stats), C.POINTER(rthx_sparse_stats)]
    L.rthx_trace_exchange_device.restype = C.c_int
    L.rthx_trace_exchange_device.argtypes = [C.c_void_p, C.POINTER(rthx_trace_args), C.c_void_p, C.c_void_p,
                                             C.c_void_p, C.c_int, C.POINTER(rthx_stats)]
    L.rthx_trace_exchange_multi.restype = C.c_int
    L.rthx_trace_exchange_multi.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.POINTER(rthx_trace_args), c_u64p,
                                            c_u64p, C.POINTER(rthx_rec_out), C.POINTER(rthx_stats)]
    L.rthx_shared_alloc.restype = C.c_int
    L.rthx_shared_alloc.argtypes = [C.c_int, C.c_uint64, C.POINTER(C.c_void_p), C.POINTER(C.c_ubyte)]
    L.rthx_shared_open.restype = C.c_int
    L.rthx_shared_open.argtypes = [C.c_int, C.POINTER(C.c_ubyte), C.POINTER(C.c_void_p)]
    L.rthx_shared_close.restype = C.c_int
    L.rthx_shared_close.argtypes = [C.c_int, C.c_void_p]
    L.rthx_shared_free.restype = C.c_int
    L.rthx_shared_free.argtypes = [C.c_int, C.c_void_p]
    L.rthx_smooth_F.restype = C.c_int
    L.rthx_smooth_F.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, c_f64p, C.c_int, C.c_double, C.c_int,
                                c_f64p, C.POINTER(rthx_smooth_stats)]
    L.rthx_smooth_DkAP.restype = C.c_int
    L.rthx_smooth_DkAP.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, c_f64p, C.c_int, C.c_int, C.c_double, C.c_int,
                                   c_f64p, C.POINTER(rthx_smooth_stats)]
    L.rthx_smooth_sparse.restype = C.c_int
    L.rthx_smooth_sparse.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, c_i64p, c_i32p, c_f64p, c_f64p, C.c_int, C.c_double, C.c_int,
                                     C.POINTER(C.c_int64), C.POINTER(rthx_smooth_stats)]
    L.rthx_smooth_sparse_csc.restype = C.c_int
    L.rthx_smooth_sparse_csc.argtypes = [C.c_void_p, C.c_int, C.c_int, c_i64p, C.c_void_p, c_f64p]
    L.rthx_solve_grey.restype = C.c_int
    L.rthx_solve_grey.argtypes = [C.c_void_p, C.POINTER(rthx_solve_args), c_f64p, c_f64p, C.POINTER(rthx_solve_stats)]
    L.rthx_release_cached.restype = C.c_int
    L.rthx_release_cached.argtypes = []
    L.rthx_counts_nnz.restype = C.c_int
    L.rthx_counts_nnz.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_int64)]
    L.rthx_counts_csr.restype = C.c_int
    L.rthx_counts_csr.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_int64), c_i32p, c_u64p, c_f64p]
    L.rthx_counts_stats.restype = C.c_int
    L.rthx_counts_stats.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_double)]
    L.rthx_counts_csc.restype = C.c_int
    L.rthx_counts_csc.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int64), C.c_void_p, c_u64p, c_f64p]
    L.rthx_flag_signal.restype = C.c_int
    L.rthx_flag_signal.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p]
    L.rthx_flag_wait.restype = C.c_int
    L.rthx_flag_wait.argtypes = [C.c_void_p, C.c_int, C.c_uint64, C.c_double, C.c_void_p, C.c_void_p]
    L.rthx_host_register.restype = C.c_int
    L.rthx_host_register.argtypes = [C.c_void_p, C.c_uint64]
    L.rthx_host_unregister.restype = C.c_int
    L.rthx_host_unregister.argtypes = [C.c_void_p]
    L.rthx_set_copy_helpers.restype = C.c_int
    L.rthx_set_copy_helpers.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.c_int]
    L.rthx_host_alloc.restype = C.c_int
    L.rthx_host_alloc.argtypes = [C.POINTER(C.c_void_p), C.c_uint64]
    L.rthx_host_free.restype = C.c_int
    L.rthx_host_free.argtypes = [C.c_void_p]
    L.rthx_measure_fp64_peak.restype = C.c_int
    L.rthx_measure_fp64_peak.argtypes = [C.c_void_p, C.POINTER(C.c_double)]
    L.rthx_last_error.restype = C.c_char_p
    L.rthx_last_error.argtypes = [C.c_void_p]
    L.rthx_version.restype = C.c_int
    L.rthx_version.argtypes = []
    _LIB = L
    return L


def device_count() -> int:
    """Number of usable CUDA devices as the library sees them (rthx_device_count); raises without one — no CPU fallback."""
    L = load_library()
    n = C.c_int(0)
    rc = L.rthx_device_count(C.byref(n))
    if rc != 0:
        msg = L.rthx_last_error(None)
        raise RthxError(f"rthx_device_count failed ({rc}): {msg.decode() if msg else ''}")
    return n.value


def make_trace_args(rays_per_emitter: int, seed: int = DEFAULT_SEED, bins: Sequence[int] = (0,),
                    nudge: Optional[float] = None, rec_ids: Optional[Sequence[int]] = None, rec_bin: int = 0,
                    ray_id_offset: int = 0, emitter_rank: int = 0, emitter_world: int = 1,
                    locator: int = RTHX_LOCATOR_AUTO, block_threads: int = 0, row_chunks: int = 0,
                    mode: int = RTHX_FIRST_INTERACTION):
    """Build an rthx_trace_args; returns (args, keepalive) — keep `keepalive` referenced during the call."""
    a = rthx_trace_args()
    a.rays_per_emitter = int(rays_per_emitter)
    a.ray_id_offset = int(ray_id_offset)
    a.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    a.nudge = DEFAULT_NUDGE if nudge is None else float(nudge)
    bins_arr = np.ascontiguousarray(bins, dtype=np.int32)
    a.n_bins = len(bins_arr)
    a.bins = bins_arr.ctypes.data_as(c_i32p)
    a.mode = int(mode)
    a.locator = int(locator)
    a.emitter_rank = int(emitter_rank)
    a.emitter_world = int(emitter_world)
    rec_arr = np.ascontiguousarray(rec_ids if rec_ids else [], dtype=np.int32)
    a.n_rec_ids = len(rec_arr)
    a.rec_ids = rec_arr.ctypes.data_as(c_i32p) if len(rec_arr) else None
    a.rec_bin = int(rec_bin)
    a.block_threads = int(block_threads)
    a.row_chunks = int(row_chunks)
    return a, (bins_arr, rec_arr)


class _PinnedPool:
    """Page-locked host buffers (rthx_host_alloc) for large result arrays.  cudaHostAlloc pins pages at ~1-2 GB/s, so a 900 MB
    matrix costs more to allocate than to trace; buffers return here when their numpy array is garbage-collected and are
    handed out again (best fit), up to `limit` bytes parked."""

    def __init__(self, limit: int = 8 << 30):
        self.free = []          # (capacity, address)
        self.limit = limit

    def take(self, nbytes: int):
        nbytes = max(int(nbytes), 64)
        best = None
        for k, (cap, _) in enumerate(self.free):
            if cap >= nbytes and (best is None or cap < self.free[best][0]) and cap <= 2 * nbytes + (1 << 20):
                best = k
        if best is not None:
            return self.free.pop(best)
        p = C.c_void_p()
        L = load_library()
        if L.rthx_host_alloc(C.byref(p), nbytes) != 0:
            msg = L.rthx_last_error(None)
            raise RthxError(f"rthx_host_alloc({nbytes}) failed: {msg.decode() if msg else ''}")
        return nbytes, p.value

    def give(self, cap: int, addr: int):
        if sum(c for c, _ in self.free) + cap <= self.limit:
            self.free.append((cap, addr))
        else:
            load_library().rthx_host_free(C.c_void_p(addr))

    def release(self):
        L = load_library()
        for _, addr in self.free:
            L.rthx_host_free(C.c_void_p(addr))
        self.free = []


_PINNED = _PinnedPool()


def pinned_empty(shape, dtype=np.float64) -> np.ndarray:
    """numpy array in page-locked host memory (device->host copies into it run by DMA, no staging pass)."""
    import weakref
    shape = (int(shape),) if np.isscalar(shape) else tuple(int(x) for x in shape)
    n = int(np.prod(shape)) if len(shape) else 1
    nbytes = n * np.dtype(dtype).itemsize
    cap, addr = _PINNED.take(nbytes)
    buf = (C.c_char * max(nbytes, 1)).from_address(addr)
    arr = np.frombuffer(buf, dtype=dtype, count=n).reshape(shape)
    weakref.finalize(buf, _PINNED.give, cap, addr)
    return arr


def release_pinned():
    _PINNED.release()


class DeviceTracer:
    """Owns one `rthx_handle` (mesh resident on one GPU)."""

    def __init__(self, flat, device: int = 0, _handle=None):
        self._L = load_library()
        self.flat = flat
        self.device = int(device)
        if _handle is not None:
            h = _handle
        else:
            h = C.c_void_p()
            rc = self._L.rthx_create(C.byref(h), C.byref(flat.c), self.device)
            if rc != 0:
                msg = self._L.rthx_last_error(None)
                raise RthxError(f"rthx_create failed ({rc}): {msg.decode() if msg else ''}")
        self._h = h
        info = rthx_info()
        self._check(self._L.rthx_get_info(self._h, C.byref(info)))
        self.info = info.as_dict()
        self.n_elements = info.n_elements
        self._resident = None          # the trace whose counts the library keeps on the device (_set_resident)

    def _check(self, rc: int):
        if rc != 0:
            msg = self._L.rthx_last_error(self._h)
            raise RthxError(f"rthx call failed ({rc}): {msg.decode() if msg else ''}")

    def close(self):
        if getattr(self, "_h", None):
            self._L.rthx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def trace(self, rays_per_emitter: int, counts_out: Optional[np.ndarray] = None, dense: bool = True, **kw):
        """Blocking trace with host outputs (rthx_trace_exchange).  Returns a dict with counts [nb,N,N] u64,
        lost [nb,N] u64, stats, and origins/endpoints when rec_ids is given.  dense=False leaves the counts on the
        device (counts is None): read them with `counts_csr()` or smooth them with `smooth()`."""
        rec_ids = kw.get("rec_ids")
        args, keep = make_trace_args(rays_per_emitter, **kw)
        N, nb = self.n_elements, args.n_bins
        if not dense:
            counts = None
        elif counts_out is not None:
            counts = counts_out
        elif args.emitter_world > 1:   # rows of other ranks are left untouched by the library: start from zeros when sharded
            counts = np.zeros((nb, N, N), np.uint64)
        else:                          # page-locked for anything large: the pipelined row copies then run by DMA behind the kernels
            counts = pinned_empty((nb, N, N), np.uint64) if nb * N * N > (1 << 16) else np.empty((nb, N, N), np.uint64)
        assert counts is None or (counts.dtype == np.uint64 and counts.size == nb * N * N and counts.flags["C_CONTIGUOUS"])
        lost = np.empty((nb, N), np.uint64)
        st = rthx_stats()
        rec, origins, endpoints = _recorder(rec_ids, rays_per_emitter)
        self._check(self._L.rthx_trace_exchange(self._h, C.byref(args), counts.ctypes.data_as(c_u64p) if counts is not None else None,
                                                lost.ctypes.data_as(c_u64p), C.byref(rec) if rec else None,
                                                C.byref(st)))
        self._set_resident(rays_per_emitter, kw, len(range(args.emitter_rank, N, args.emitter_world)))   # rows e = rank + y * world
        return _recorded(dict(counts=counts.reshape(nb, N, N) if counts is not None else None, lost=lost, stats=st.as_dict()), rec, origins, endpoints)

    def trace_rows(self, emitters, rays_per_emitter: int, dense: bool = True, **kw):
        """Blocking trace of the emitter rows `emitters` only (rthx_trace_exchange_rows): element indices, strictly ascending, in [0, N).
        Row y of the result is element emitters[y], equal bit for bit to that row of `trace()` with the same keywords.  Returns the dict
        of `trace()` with counts [nb, R, N] (None with dense=False: the R rows stay on the device for `counts_csr()` (R rows),
        `counts_csc()` / `counts_stats()` (the N x N matrix whose other rows are empty), `smooth()` / `smooth_sparse()` with a crop n
        whose rows are all listed, and `trace_continue()`); lost [nb, N] is 0 for unlisted elements."""
        rows = np.ascontiguousarray(emitters, dtype=np.int32).ravel()
        args, keep = make_trace_args(rays_per_emitter, **kw)
        N, nb, R = self.n_elements, args.n_bins, len(rows)
        if not dense:
            counts = None
        else:
            counts = pinned_empty((nb, R, N), np.uint64) if nb * R * N > (1 << 16) else np.empty((nb, R, N), np.uint64)
        lost = np.empty((nb, N), np.uint64)
        st = rthx_stats()
        rec, origins, endpoints = _recorder(kw.get("rec_ids"), rays_per_emitter)
        self._check(self._L.rthx_trace_exchange_rows(self._h, C.byref(args), rows.ctypes.data_as(c_i32p), R,
                                                     counts.ctypes.data_as(c_u64p) if counts is not None else None,
                                                     lost.ctypes.data_as(c_u64p), C.byref(rec) if rec else None, C.byref(st)))
        self._set_resident(rays_per_emitter, kw, R)
        return _recorded(dict(counts=counts.reshape(nb, R, N) if counts is not None else None, lost=lost, stats=st.as_dict()), rec, origins, endpoints)

    def trace_direct(self, sources, rays, reemit, bundle_energy, specular: bool = False, redirected: bool = False, sparse: bool = False, **kw):
        """method=:direct on the device (rthx_trace_direct): source y = element sources[y] (strictly ascending) traces rays[y] bundles of
        energy bundle_energy[y] through the MULTI_BOUNCE events (specular=True: mirror reflection); a bundle absorbed by element k with
        reemit[k] is emitted again from k.  Keywords of `trace()` (seed, nudge, locator, block_threads, row_chunks, ray_id_offset).
        Returns dict(absorbed [N] f64 = sum_y bundle_energy[y] counts[y][k] in ascending y, lost [N] u64 per source element,
        events, stats).  The counts stay resident as the listed rows of a rows trace (`counts_csr()`: R = len(sources) rows).
        redirected=True (rthx_trace_direct_fields) also tallies every scattering and reflection at element k in a second count block,
        read out with `counts_csr(bin=1)`, and adds redirected [N] f64, the same fixed-order sum over that block; everything else is
        bit for bit the result of redirected=False.
        sparse=True (rthx_trace_direct_sparse) tallies the counts into the hashed row tally instead of dense [R][N] rows, for source
        lists whose 8 R N bytes (16 R N with redirected=True) do not fit; every result and read-out is bit for bit that of sparse=False,
        and the dict adds `sparse_stats` (pairs, flushes, row groups)."""
        from ._abi import RTHX_MULTI_BOUNCE, RTHX_MULTI_BOUNCE_SPECULAR
        rows = np.ascontiguousarray(sources, dtype=np.int32).ravel()
        R, N = len(rows), self.n_elements
        nr = np.ascontiguousarray(rays, dtype=np.int64).ravel()
        re_ = np.ascontiguousarray(reemit, dtype=np.uint8).ravel()
        w = np.ascontiguousarray(bundle_energy, dtype=np.float64).ravel()
        if len(nr) != R or len(w) != R or len(re_) != N:
            raise ValueError(f"trace_direct: rays and bundle_energy need {R} entries (one per source), reemit {N} (one per element)")
        args, keep = make_trace_args(0, mode=RTHX_MULTI_BOUNCE_SPECULAR if specular else RTHX_MULTI_BOUNCE, **kw)
        absorbed = np.empty(N, np.float64)
        red = np.empty(N, np.float64) if redirected else None
        lost = np.empty(N, np.uint64)
        events = C.c_int64(0)
        st = rthx_stats()
        head = (self._h, C.byref(args), rows.ctypes.data_as(c_i32p), nr.ctypes.data_as(c_i64p), R, re_.ctypes.data_as(C.POINTER(C.c_uint8)),
                w.ctypes.data_as(c_f64p), absorbed.ctypes.data_as(c_f64p))
        tail = (lost.ctypes.data_as(c_u64p), C.byref(events), C.byref(st))
        sst = rthx_sparse_stats()
        if sparse:
            self._check(self._L.rthx_trace_direct_sparse(*head, red.ctypes.data_as(c_f64p) if redirected else None, *tail, C.byref(sst)))
        elif redirected:
            self._check(self._L.rthx_trace_direct_fields(*head, red.ctypes.data_as(c_f64p), *tail))
        else:
            self._check(self._L.rthx_trace_direct(*head, *tail))
        self._resident = dict(kw={}, hi=0, sparse=bool(sparse), rows=R)
        out = dict(absorbed=absorbed, lost=lost, events=int(events.value), stats=st.as_dict())
        if redirected:
            out["redirected"] = red
        if sparse:
            out["sparse_stats"] = sst.as_dict()
        return out

    def trace_sparse(self, rays_per_emitter: int, **kw):
        """Blocking trace with the hashed row tally (rthx_trace_exchange_sparse): the counts never exist in dense form and stay on
        the device as sorted (row, column, total) triplets, so device memory is O(non-zeros).  Same keywords and result as
        `trace(dense=False)` (counts is None; `counts_csr()`, `counts_csc()`, `counts_stats()` and `smooth_sparse()` read the
        resident counts and return what they return after it, bit for bit), plus `sparse_stats` (pairs, flushes, row groups).
        FIRST_INTERACTION only."""
        args, keep = make_trace_args(rays_per_emitter, **kw)
        lost = np.empty((args.n_bins, self.n_elements), np.uint64)
        st, sst = rthx_stats(), rthx_sparse_stats()
        rec, origins, endpoints = _recorder(kw.get("rec_ids"), rays_per_emitter)
        self._check(self._L.rthx_trace_exchange_sparse(self._h, C.byref(args), lost.ctypes.data_as(c_u64p), C.byref(rec) if rec else None,
                                                       C.byref(st), C.byref(sst)))
        self._set_resident(rays_per_emitter, kw, len(range(args.emitter_rank, self.n_elements, args.emitter_world)), sparse=True)
        return _recorded(dict(counts=None, lost=lost, stats=st.as_dict(), sparse_stats=sst.as_dict()), rec, origins, endpoints)

    # keywords that fix the resident trace's ray stream; trace_continue repeats them unless given
    _STREAM_KW = ("seed", "bins", "nudge", "mode", "locator", "emitter_rank", "emitter_world")

    def _set_resident(self, rays_per_emitter: int, kw, rows: int, sparse: bool = False):
        """Record the trace whose counts the library now keeps on the device: its stream keywords and the end of its ray-id range (what
        trace_continue repeats and continues), its form, and its rows per bin (the R of counts_csr)."""
        lo = int(kw.get("ray_id_offset", 0))
        self._resident = dict(kw={k: kw[k] for k in self._STREAM_KW if k in kw}, hi=lo + int(rays_per_emitter), sparse=sparse, rows=int(rows))

    def trace_continue(self, rays_per_emitter: int, **kw):
        """Add `rays_per_emitter` rays per owned emitter to the counts resident from the last `trace(dense=False)`, `trace_sparse()` or
        `trace_continue()` (rthx_trace_exchange_continue), in their dense or hashed form.  The seed, bins, nudge, mode, locator and
        shard of that trace are repeated unless given (the library rejects any that differ), and ray_id_offset is the end of the
        resident ray-id range.  Afterwards every read-out of the resident counts equals, bit for bit, the read-out after ONE trace of
        the whole range.  Returns the dict of the trace that left the counts resident (sparse_stats after a hashed one), with lost
        cumulative over the whole range; origins / endpoints hold this call's recorded rays."""
        res = self._resident or dict(kw={}, hi=0, sparse=False)
        kw = {**res["kw"], "ray_id_offset": res["hi"], **kw}
        args, keep = make_trace_args(rays_per_emitter, **kw)
        lost = np.empty((args.n_bins, self.n_elements), np.uint64)
        st, sst = rthx_stats(), rthx_sparse_stats()
        rec, origins, endpoints = _recorder(kw.get("rec_ids"), rays_per_emitter)
        self._check(self._L.rthx_trace_exchange_continue(self._h, C.byref(args), lost.ctypes.data_as(c_u64p), C.byref(rec) if rec else None,
                                                         C.byref(st), C.byref(sst)))
        res["hi"] = int(args.ray_id_offset) + int(rays_per_emitter)
        out = dict(counts=None, lost=lost, stats=st.as_dict())
        if res["sparse"]:
            out["sparse_stats"] = sst.as_dict()
        return _recorded(out, rec, origins, endpoints)

    def trace_device(self, rays_per_emitter: int, counts_ptr: int, lost_ptr: int, stream: int = 0,
                     zero_first=True, **kw):
        """Asynchronous trace into device buffers (rthx_trace_exchange_device); pointers are raw device addresses
        (e.g. torch.Tensor.data_ptr()), stream a cudaStream_t handle (e.g. torch.cuda.current_stream().cuda_stream)."""
        args, keep = make_trace_args(rays_per_emitter, **kw)
        st = rthx_stats()
        self._check(self._L.rthx_trace_exchange_device(self._h, C.byref(args), C.c_void_p(counts_ptr),
                                                       C.c_void_p(lost_ptr), C.c_void_p(stream),
                                                       int(zero_first), C.byref(st)))
        return st.as_dict()

    def counts_csr(self, bin: int = 0, values: bool = True, normalised: bool = True):
        """CSR read-out of the counts resident on the device (rthx_counts_nnz / rthx_counts_csr): returns
        (row_ptr [R+1] i64, cols [nnz] i32, counts [nnz] u64 or None, F_vals [nnz] f64 = count/row total or None); R = N after a
        plain trace, the number of owned rows (elements rank + y * world) after a sharded one, the listed rows after `trace_rows()`.
        After `trace_direct()` bin 0 holds the absorption counts of the sources, and with redirected=True bin 1 their redirections."""
        nnz = C.c_int64(0)
        self._check(self._L.rthx_counts_nnz(self._h, int(bin), C.byref(nnz)))
        N, k = self.n_elements, max(1, nnz.value)
        R = self._resident["rows"] if self._resident else N
        row_ptr = np.empty(R + 1, np.int64)
        cols = np.empty(k, np.int32)
        vals = np.empty(k, np.uint64) if values else None
        fv = np.empty(k, np.float64) if normalised else None
        self._check(self._L.rthx_counts_csr(self._h, int(bin), row_ptr.ctypes.data_as(C.POINTER(C.c_int64)), cols.ctypes.data_as(c_i32p),
                                            vals.ctypes.data_as(c_u64p) if values else None,
                                            fv.ctypes.data_as(c_f64p) if normalised else None))
        n = nnz.value
        return row_ptr, cols[:n], (vals[:n] if values else None), (fv[:n] if normalised else None)

    def set_copy_helpers(self, others: Sequence["DeviceTracer"]):
        """Let large device->host result copies of this tracer (CSC arrays, F_smooth) use the PCIe links of the tracers on the other
        devices as well (rthx_set_copy_helpers); an empty list clears the registration."""
        hs = (C.c_void_p * max(1, len(others)))(*[t._h for t in others])
        self._check(self._L.rthx_set_copy_helpers(self._h, hs, len(others)))
        self._copy_helpers = list(others)          # keep them alive

    def counts_stats(self, bin: int = 0):
        """(nnz, chi) of the counts resident on the device: non-zeros and the surface-gas cross-coupling of the
        row-normalised F (cross_coupling_chi, smoothExchangeFactors.jl:212-241) — rthx_counts_stats."""
        nnz, chi = C.c_int64(0), C.c_double(0.0)
        self._check(self._L.rthx_counts_stats(self._h, int(bin), C.byref(nnz), C.byref(chi)))
        return nnz.value, chi.value

    def counts_csc(self, bin: int = 0, values: bool = False, normalised: bool = True, index64: bool = False, index_base: int = 0,
                   pinned: bool = True):
        """CSC read-out of the counts resident on the device (rthx_counts_csc): (colptr [N+1] i64, rowval [nnz] i32 | i64,
        counts [nnz] u64 or None, F_vals [nnz] f64 = count / row total or None) — the three arrays of the reference's
        SparseMatrixCSC, rows ascending within each column."""
        nnz, _ = self.counts_stats(bin)
        N, k = self.n_elements, max(1, nnz)
        alloc = pinned_empty if pinned and k > (1 << 16) else (lambda shape, dtype: np.empty(shape, dtype))
        colptr = np.empty(N + 1, np.int64)
        rowval = alloc(k, np.int64 if index64 else np.int32)
        vals = alloc(k, np.uint64) if values else None
        fv = alloc(k, np.float64) if normalised else None
        self._check(self._L.rthx_counts_csc(self._h, int(bin), int(index_base), 1 if index64 else 0,
                                            colptr.ctypes.data_as(C.POINTER(C.c_int64)), rowval.ctypes.data_as(C.c_void_p),
                                            vals.ctypes.data_as(c_u64p) if values else None,
                                            fv.ctypes.data_as(c_f64p) if normalised else None))
        return colptr, rowval[:nnz], (vals[:nnz] if values else None), (fv[:nnz] if normalised else None)

    def smooth(self, w, n: Optional[int] = None, counts: Optional[np.ndarray] = None, F: Optional[np.ndarray] = None,
               bin: int = 0, max_iters: int = 1000, target: float = 0.0, measure_pass: bool = False,
               out: Optional[np.ndarray] = None, k_dykstra: int = 0):
        """Dense reciprocity smoothing on the device (rthx_smooth_DkAP: `k_dykstra` Dykstra rounds, then AP).  Source: `counts` (u64 [n,n]) or `F` (f64 [n,n])
        from the host, or — with neither — the counts of traced bin `bin` still resident from the last `trace()`.
        `w` must already be renormalised (w / min(w)).  Returns (F_smooth [n,n] f64, stats dict)."""
        w = np.ascontiguousarray(w, dtype=np.float64)
        n = len(w) if n is None else int(n)
        assert len(w) == n
        self._resident_F = None        # whatever F_smooth an earlier call left on the device is about to be replaced
        if counts is not None:
            src = np.ascontiguousarray(counts, dtype=np.uint64); assert src.shape == (n, n)
            source, ptr = RTHX_SMOOTH_FROM_COUNTS, src.ctypes.data_as(C.c_void_p)
        elif F is not None:
            src = np.ascontiguousarray(F, dtype=np.float64); assert src.shape == (n, n)
            source, ptr = RTHX_SMOOTH_FROM_F, src.ctypes.data_as(C.c_void_p)
        else:
            src, source, ptr = None, RTHX_SMOOTH_FROM_LAST_TRACE, None
        F_out = out if out is not None else (pinned_empty((n, n), np.float64) if n * n > (1 << 16) else np.empty((n, n), np.float64))
        assert F_out.dtype == np.float64 and F_out.size == n * n and F_out.flags["C_CONTIGUOUS"]
        st = rthx_smooth_stats()
        self._check(self._L.rthx_smooth_DkAP(self._h, source, ptr, int(bin), n, w.ctypes.data_as(c_f64p), int(k_dykstra),
                                             int(max_iters), float(target), 1 if measure_pass else 0,
                                             F_out.ctypes.data_as(c_f64p), C.byref(st)))
        return F_out.reshape(n, n), st.as_dict()

    def smooth_sparse(self, w, n: Optional[int] = None, F=None, bin: int = 0, max_iters: int = 1000, target: float = 0.0,
                      measure_pass: bool = False):
        """Sparse reciprocity smoothing on the device (rthx_smooth_sparse: AP on the union pattern of F and F', the sparse branch
        of smooth_F).  Source: `F`, a scipy.sparse matrix (sent as CSC; its rows must be sorted within each column), or — without
        it — the counts of traced bin `bin` still resident from the last `trace()`, cropped to the leading n x n block.  `w` must
        already be renormalised (w / min(w)).  Returns (F_smooth as scipy.sparse.csc_matrix over page-locked arrays, stats dict)."""
        import scipy.sparse as sp
        w = np.ascontiguousarray(w, dtype=np.float64)
        n = len(w) if n is None else int(n)
        assert len(w) == n
        self._resident_F = None        # a dense F_smooth an earlier smooth() left on the device is replaced
        keep = (None, None, None)
        source = RTHX_SMOOTH_FROM_LAST_TRACE
        if F is not None:
            Fc = F.tocsc() if sp.issparse(F) else sp.csc_matrix(F)
            assert Fc.shape == (n, n)
            keep = (np.ascontiguousarray(Fc.indptr, dtype=np.int64), np.ascontiguousarray(Fc.indices, dtype=np.int32),
                    np.ascontiguousarray(Fc.data, dtype=np.float64))
            source = RTHX_SMOOTH_FROM_CSC
        ptrs = [a.ctypes.data_as(t) if a is not None else None for a, t in zip(keep, (c_i64p, c_i32p, c_f64p))]
        nnz = C.c_int64(0)
        st = rthx_smooth_stats()
        self._check(self._L.rthx_smooth_sparse(self._h, source, int(bin), n, *ptrs, w.ctypes.data_as(c_f64p), int(max_iters),
                                               float(target), 1 if measure_pass else 0, C.byref(nnz), C.byref(st)))
        nz = nnz.value
        k = max(1, nz)
        alloc = pinned_empty if k > (1 << 16) else (lambda shape, dtype: np.empty(shape, dtype))
        colptr = np.empty(n + 1, np.int64)
        rowval = alloc(k, np.int32 if nz < 2 ** 31 else np.int64)
        nzval = alloc(k, np.float64)
        self._check(self._L.rthx_smooth_sparse_csc(self._h, 0, 0 if nz < 2 ** 31 else 1, colptr.ctypes.data_as(c_i64p),
                                                   rowval.ctypes.data_as(C.c_void_p), nzval.ctypes.data_as(c_f64p)))
        if nz < 2 ** 31:
            colptr = colptr.astype(np.int32)           # scipy wants one index type; N + 1 entries, the big array stays as it is
        Fs = sp.csc_matrix((nzval[:nz], rowval[:nz], colptr), shape=(n, n), copy=False)
        Fs.has_sorted_indices = True                   # rows ascend within each column by construction
        return Fs, st.as_dict()

    def solve_grey(self, coeff, rhs, F=None, col_major: bool = False, memory: int = 50, max_iters: int = 0,
                   rtol: float = 1e-12, atol: float = -1.0, measure_pass: bool = False):
        """(I - diag(coeff) F') j = rhs by restarted GMRES on the device (rthx_solve_grey).  `F`: None — the F_smooth
        still resident on the device from the last `smooth()`; a dense [n,n] float64 array (C order, or the memory of a
        column-major matrix with col_major=True); or a scipy.sparse matrix (converted to CSC, the reference's
        SparseMatrixCSC).  Returns (j [n], g = F'j [n], stats dict)."""
        import scipy.sparse as sp
        coeff = np.ascontiguousarray(coeff, dtype=np.float64)
        rhs = np.ascontiguousarray(rhs, dtype=np.float64)
        n = len(rhs)
        assert len(coeff) == n
        a = rthx_solve_args()
        a.n, a.memory, a.max_iters, a.measure_pass = n, int(memory), int(max_iters), 1 if measure_pass else 0
        a.rtol, a.atol = float(rtol), float(atol)
        a.coeff, a.rhs = coeff.ctypes.data_as(c_f64p), rhs.ctypes.data_as(c_f64p)
        keep = None
        if F is None:
            a.source = RTHX_SOLVE_FROM_LAST_SMOOTH
        elif sp.issparse(F):
            Fc = F.tocsc()
            Fc.sort_indices()
            assert Fc.shape == (n, n)
            keep = (np.ascontiguousarray(Fc.indptr, dtype=np.int64), np.ascontiguousarray(Fc.indices, dtype=np.int32),
                    np.ascontiguousarray(Fc.data, dtype=np.float64))
            a.source = RTHX_SOLVE_FROM_CSC
            a.colptr, a.rowval, a.nzval = (keep[0].ctypes.data_as(c_i64p), keep[1].ctypes.data_as(c_i32p),
                                           keep[2].ctypes.data_as(c_f64p))
        else:
            keep = np.ascontiguousarray(F, dtype=np.float64)
            assert keep.shape == (n, n)
            a.source, a.layout = RTHX_SOLVE_FROM_DENSE, (RTHX_COL_MAJOR if col_major else RTHX_ROW_MAJOR)
            a.F_dense = keep.ctypes.data_as(c_f64p)
        j = np.empty(n)
        g = np.empty(n)
        st = rthx_solve_stats()
        self._check(self._L.rthx_solve_grey(self._h, C.byref(a), j.ctypes.data_as(c_f64p), g.ctypes.data_as(c_f64p), C.byref(st)))
        return j, g, st.as_dict()

    def measure_fp64_peak(self) -> float:
        v = C.c_double(0.0)
        self._check(self._L.rthx_measure_fp64_peak(self._h, C.byref(v)))
        return v.value


def _recorder(rec_ids, rays_per_emitter: int):
    """rthx_rec_out over fresh host arrays for `rec_ids` (None when recording is off): (rec, origins, endpoints)."""
    if not rec_ids:
        return None, None, None
    cap = len(rec_ids) * int(rays_per_emitter)
    origins = np.zeros((max(cap, 1), 2))
    endpoints = np.zeros((max(cap, 1), 2))
    return rthx_rec_out(cap, origins.ctypes.data_as(c_f64p), endpoints.ctypes.data_as(c_f64p), 0), origins, endpoints


def _recorded(out, rec, origins, endpoints):
    """`out` with the rays the recorder caught (origins / endpoints of _recorder's arrays) when recording was on."""
    if rec is not None:
        out["origins"] = origins[: rec.n_recorded].copy()
        out["endpoints"] = endpoints[: rec.n_recorded].copy()
    return out


def create_multi(flat, devices: Sequence[int]):
    """One DeviceTracer per device from ONE host-side mesh preparation (rthx_create_multi)."""
    L = load_library()
    devs = [int(d) for d in devices]
    hs = (C.c_void_p * len(devs))()
    ids = (C.c_int * len(devs))(*devs)
    rc = L.rthx_create_multi(hs, C.byref(flat.c), ids, len(devs))
    if rc != 0:
        msg = L.rthx_last_error(None)
        raise RthxError(f"rthx_create_multi failed ({rc}): {msg.decode() if msg else ''}")
    return [DeviceTracer(flat, device=d, _handle=C.c_void_p(hs[i])) for i, d in enumerate(devs)]


def trace_multi(tracers: Sequence[DeviceTracer], rays_per_emitter: int, counts_out: Optional[np.ndarray] = None, dense: bool = True, **kw):
    """Single-process multi-GPU trace (rthx_trace_exchange_multi).  dense=True: every device copies its rows into the host
    matrix `counts_out` (allocated page-locked when not given).  dense=False: the devices flush their rows into one matrix on
    tracers[0]'s device over NVLink peer memory; it stays resident there (counts is None) for `tracers[0].counts_csc()` /
    `.counts_csr()` / `.smooth()`."""
    L = load_library()
    rec_ids = kw.get("rec_ids")
    args, keep = make_trace_args(rays_per_emitter, **kw)
    N, nb = tracers[0].n_elements, args.n_bins
    if not dense:
        counts = None
    elif counts_out is not None:
        counts = counts_out
    else:
        counts = pinned_empty((nb, N, N), np.uint64)
    assert counts is None or (counts.dtype == np.uint64 and counts.size == nb * N * N and counts.flags["C_CONTIGUOUS"])
    lost = np.empty((nb, N), np.uint64)
    st = rthx_stats()
    hs = (C.c_void_p * len(tracers))(*[t._h for t in tracers])
    rec, origins, endpoints = _recorder(rec_ids, rays_per_emitter)
    rc = L.rthx_trace_exchange_multi(hs, len(tracers), C.byref(args), counts.ctypes.data_as(c_u64p) if counts is not None else None,
                                     lost.ctypes.data_as(c_u64p), C.byref(rec) if rec else None, C.byref(st))
    if rc != 0:
        msg = L.rthx_last_error(tracers[0]._h)
        raise RthxError(f"rthx_trace_exchange_multi failed ({rc}): {msg.decode() if msg else ''}")
    tracers[0]._set_resident(rays_per_emitter, kw, N)
    return _recorded(dict(counts=counts.reshape(nb, N, N) if counts is not None else None, lost=lost, stats=st.as_dict()), rec, origins, endpoints)


def merge_row_tiles(tiles, N: int, n_bins: int, tile_rows=None):
    """Merge the CSR read-outs of interleaved row tiles (tile t holds the rows e = t (mod n_tiles), in order, or with `tile_rows` the
    ascending elements tile_rows[t]; rows no tile holds stay empty) into one CSR matrix per traced bin.  tiles[t][k] = (row_ptr, cols,
    F_vals) of bin k.  Returns a list of (row_ptr [N+1], cols, F_vals)."""
    n_tiles = len(tiles)
    if tile_rows is None:
        tile_rows = [np.arange(t, N, n_tiles) for t in range(n_tiles)]
    mats = []
    for k in range(n_bins):
        nnz_row = np.zeros(N, np.int64)
        for t in range(n_tiles):
            nnz_row[tile_rows[t]] = np.diff(tiles[t][k][0])
        row_ptr = np.zeros(N + 1, np.int64)
        np.cumsum(nnz_row, out=row_ptr[1:])
        cols = np.empty(int(row_ptr[-1]), np.int32)
        vals = np.empty(int(row_ptr[-1]), np.float64)
        for t in range(n_tiles):
            rp, c_t, f_t = tiles[t][k]
            rows = tile_rows[t]
            lens = np.diff(rp)
            # destination of every entry of the tile: start of its global row + offset inside the row
            dst = np.repeat(row_ptr[rows] - rp[:-1], lens) + np.arange(int(rp[-1]), dtype=np.int64)
            cols[dst] = c_t
            vals[dst] = f_t
        mats.append((row_ptr, cols, vals))
    return mats


def _tile_readout(tracer: DeviceTracer, n_bins: int, divide: bool = False):
    """(per-bin CSR pieces, per-bin chi share) of the rows resident on `tracer` after a sharded trace.  F = count * (1 / row total)
    as rthx_counts_csr forms it, or with `divide` count / row total as rthx_counts_csc does (IEEE division of exact integers: the
    same bits as the device's CSC read-out of an unsharded trace)."""
    parts, chi = [], np.zeros(n_bins)
    for k in range(n_bins):
        chi[k] = tracer.counts_stats(k)[1]
        if divide:
            rp, cols, vals, _ = tracer.counts_csr(k, values=True, normalised=False)
            cs = np.zeros(len(vals) + 1, np.uint64)
            np.cumsum(vals, out=cs[1:])
            total = cs[rp[1:]] - cs[rp[:-1]]
            fv = vals.astype(np.float64) / np.repeat(total, np.diff(rp)).astype(np.float64)
        else:
            rp, cols, _, fv = tracer.counts_csr(k, values=False, normalised=True)
        parts.append((rp, cols.copy(), fv.copy()))
    return parts, chi


def trace_row_tiles(tracer: DeviceTracer, rays_per_emitter: int, n_tiles: int, **kw):
    """Exchange factors of a mesh whose dense 8 N^2-byte count matrix does not fit (N >> 57 k elements, SURVEY.md section 5): the
    emitter rows are traced in `n_tiles` interleaved tiles (rows e = t (mod n_tiles) — the multi-GPU partition, run in sequence on
    one device), each tile's counts stay on the device and only their non-zeros come back (rthx_counts_csr); the tiles are merged
    into ONE row-normalised CSR matrix.  Counts are those of the untiled trace bit for bit (the Philox stream is keyed by ray
    id and emitter).  Returns a list of (row_ptr [N+1], cols, F_vals) per traced bin, plus lost [nb, N] and chi per bin."""
    N = tracer.n_elements
    n_tiles = max(1, min(int(n_tiles), N))
    nb = len(kw.get("bins", (0,)))
    tiles = []
    lost = np.zeros((nb, N), np.uint64)
    chi = np.zeros(nb)
    for t in range(n_tiles):
        out = tracer.trace(rays_per_emitter, dense=False, emitter_rank=t, emitter_world=n_tiles, **kw)
        stats = out["stats"]
        lost += out["lost"]
        parts, c = _tile_readout(tracer, nb)
        tiles.append(parts)
        chi += c
    return dict(csr=merge_row_tiles(tiles, N, nb), lost=lost, chi=chi, stats=stats)


def trace_sparse_multi(tracers: Sequence[DeviceTracer], rays_per_emitter: int, refine: bool = False, **kw):
    """The hashed-tally trace (DeviceTracer.trace_sparse) on several devices at once: device r traces the emitters e = r (mod n)
    (one host thread per handle; the ctypes call releases the GIL), its rows stay on its device and only their non-zeros come back;
    the host merges them into ONE row-normalised CSR matrix per traced bin (merge_row_tiles).  Counts are those of a single-device
    trace bit for bit, and F = count / row total is the F_raw of a single-device trace bit for bit.  Returns dict(csr=[(row_ptr, cols, F_vals)] per bin, lost [nb, N], chi per bin, stats, sparse_stats), plus
    origins / endpoints with rec_ids: the points of device 0's recorded emitters first, then device 1's, ... (each in ascending
    (emitter, ray) order).  refine=True continues the shards left resident by the previous call (DeviceTracer.trace_continue) instead
    of tracing them afresh; lost is then cumulative."""
    from concurrent.futures import ThreadPoolExecutor
    n = len(tracers)
    N = tracers[0].n_elements
    nb = len(kw.get("bins", (0,)))
    rec_ids = kw.pop("rec_ids", None)

    def run(r):
        own = [e for e in (rec_ids or []) if e % n == r]
        trace = tracers[r].trace_continue if refine else tracers[r].trace_sparse
        out = trace(rays_per_emitter, emitter_rank=r, emitter_world=n, rec_ids=own or None, **kw)
        parts, chi = _tile_readout(tracers[r], nb, divide=True)
        return out, parts, chi

    with ThreadPoolExecutor(max_workers=n) as ex:
        res = list(ex.map(run, range(n)))
    result = _combine_shards(res, N, nb, bool(rec_ids))
    result["sparse_stats"] = {k: sum(o["sparse_stats"][k] for o, _, _ in res) for k in ("pairs", "nnz", "flushes", "row_groups")}
    return result


def trace_rows_multi(tracers: Sequence[DeviceTracer], emitters, rays_per_emitter: int, refine: bool = False, **kw):
    """The rows trace (DeviceTracer.trace_rows, counts left on the devices) of a list too large for one device, on several devices at
    once: device r traces the r-th contiguous block of the list as its own rows trace (one host thread per handle), and only their
    non-zeros come back; the host merges them into ONE row-normalised CSR matrix per traced bin over all N rows, unlisted rows empty
    (merge_row_tiles).  F = count / row total is the F_raw of a single-device rows trace bit for bit.  Returns dict(csr=[(row_ptr, cols,
    F_vals)] per bin, lost [nb, N], chi per bin, stats), plus origins / endpoints with rec_ids: the blocks ascend, so device 0's points
    followed by device 1's ... are in ascending (emitter, ray) order, as a single-device trace records them.  refine=True continues the
    rows left resident by the previous call (DeviceTracer.trace_continue)."""
    from concurrent.futures import ThreadPoolExecutor
    n = len(tracers)
    N = tracers[0].n_elements
    nb = len(kw.get("bins", (0,)))
    rec_ids = kw.pop("rec_ids", None)
    rows = np.ascontiguousarray(emitters, dtype=np.int32).ravel()
    parts_rows = np.array_split(rows, n)

    def run(r):
        own = [e for e in (rec_ids or []) if e in set(parts_rows[r].tolist())]
        if refine:
            out = tracers[r].trace_continue(rays_per_emitter, rec_ids=own or None, **kw)
        else:
            out = tracers[r].trace_rows(parts_rows[r], rays_per_emitter, dense=False, rec_ids=own or None, **kw)
        parts, chi = _tile_readout(tracers[r], nb, divide=True)
        return out, parts, chi

    live = [r for r in range(n) if len(parts_rows[r])]        # fewer rows than devices: the others stay idle
    with ThreadPoolExecutor(max_workers=len(live)) as ex:
        res = list(ex.map(run, live))
    return _combine_shards(res, N, nb, bool(rec_ids), tile_rows=[parts_rows[r] for r in live])


def _combine_shards(res, N: int, nb: int, recorded: bool, tile_rows=None):
    """One result from the per-device runs res = [(trace output, CSR pieces, chi)] of trace_sparse_multi / trace_rows_multi: the pieces
    merged into one CSR matrix per bin (merge_row_tiles), lost and chi summed, device 0's stats with the ray counts summed and the times of
    the slowest device, and with `recorded` the recorded rays of every device in device order."""
    outs = [o for o, _, _ in res]
    lost = np.zeros((nb, N), np.uint64)
    chi = np.zeros(nb)
    for out, _, c in res:
        lost += out["lost"]
        chi += c
    stats = dict(outs[0]["stats"])
    for k, agg in (("kernel_ms", max), ("total_ms", max), ("rays_traced", sum), ("rays_lost", sum)):
        stats[k] = agg(o["stats"][k] for o in outs)
    result = dict(csr=merge_row_tiles([p for _, p, _ in res], N, nb, tile_rows), lost=lost, chi=chi, stats=stats)
    if recorded:
        for k in ("origins", "endpoints"):
            result[k] = np.concatenate([o.get(k, np.zeros((0, 2))) for o in outs], axis=0)
    return result


class SharedDeviceBuffer:
    """A device buffer owned by one rank and mapped by the others through CUDA IPC (rthx_shared_alloc / _open).
    Exposes `__cuda_array_interface__` so `torch.as_tensor(buf, device=...)` gives a zero-copy int64 view."""

    def __init__(self, device: int, n_int64: int, handle: Optional[bytes] = None):
        self._L = load_library()
        self.device = int(device)
        self.n = int(n_int64)
        self.owner = handle is None
        ptr = C.c_void_p()
        if self.owner:
            hb = (C.c_ubyte * 64)()
            rc = self._L.rthx_shared_alloc(self.device, self.n * 8, C.byref(ptr), hb)
            self.handle = bytes(hb)
        else:
            hb = (C.c_ubyte * 64)(*handle)
            rc = self._L.rthx_shared_open(self.device, hb, C.byref(ptr))
            self.handle = bytes(handle)
        if rc != 0:
            msg = self._L.rthx_last_error(None)
            raise RthxError(f"shared buffer {'alloc' if self.owner else 'open'} failed ({rc}): {msg.decode() if msg else ''}")
        self.ptr = ptr.value
        self.__cuda_array_interface__ = {"shape": (self.n,), "typestr": "<i8", "data": (self.ptr, False), "version": 2,
                                         "strides": None}

    def close(self):
        if getattr(self, "ptr", None):
            (self._L.rthx_shared_free if self.owner else self._L.rthx_shared_close)(self.device, C.c_void_p(self.ptr))
            self.ptr = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class SharedHostMatrix:
    """A UInt64 count matrix in POSIX shared memory, page-locked in every process that maps it: each rank's
    `DeviceTracer.trace(..., counts_out=m.array, emitter_rank=r, emitter_world=W)` copies its own rows over its own PCIe
    link, overlapped with tracing, and rank 0 reads the assembled matrix after a barrier — no device-side gather."""

    def __init__(self, name: str, shape, create: bool):
        from multiprocessing import shared_memory, resource_tracker
        nbytes = int(np.prod(shape)) * 8
        if create:
            try:                                   # a stale segment of a crashed run
                old = shared_memory.SharedMemory(name=name, create=False)
                old.close(); old.unlink()
            except FileNotFoundError:
                pass
        self.shm = shared_memory.SharedMemory(name=name, create=create, size=nbytes)
        if not create:
            try:                                   # Python < 3.13 would unlink the segment when an attaching process exits
                resource_tracker.unregister(self.shm._name, "shared_memory")
            except Exception:
                pass
        self.owner = create
        self.array = np.ndarray(shape, dtype=np.uint64, buffer=self.shm.buf)
        L = load_library()
        self._L = L
        self.registered = L.rthx_host_register(C.c_void_p(self.array.ctypes.data), nbytes) == 0
        # not page-locked (e.g. locked-memory limit): the library's pinned staging path still serves it

    def close(self):
        if getattr(self, "shm", None) is not None:
            if self.registered:
                self._L.rthx_host_unregister(C.c_void_p(self.array.ctypes.data))
            self.array = None
            self.shm.close()
            if self.owner:
                try:
                    self.shm.unlink()
                except FileNotFoundError:
                    pass
            self.shm = None
