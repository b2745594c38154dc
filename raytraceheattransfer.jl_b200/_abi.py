"""ctypes mirror of include/rthx.h (struct layouts must stay in lock-step with the header)."""
from __future__ import annotations

import ctypes as C

RTHX_OK = 0
RTHX_FIRST_INTERACTION = 0
RTHX_MULTI_BOUNCE = 1
RTHX_MULTI_BOUNCE_SPECULAR = 2
RTHX_LOCATOR_AUTO = 0
RTHX_LOCATOR_GENERIC = 1
RTHX_ZERO_NONE, RTHX_ZERO_ALL, RTHX_ZERO_OWN_ROWS = 0, 1, 2
RTHX_DEST_PEER = 16      # OR into zero_first: the matrix lives in another device's memory (CUDA IPC mapping)

c_i32p = C.POINTER(C.c_int32)
c_f64p = C.POINTER(C.c_double)
c_u8p = C.POINTER(C.c_uint8)
c_u64p = C.POINTER(C.c_uint64)


class rthx_mesh(C.Structure):
    _fields_ = [
        ("n_coarse", C.c_int32), ("n_cells", C.c_int32), ("n_bands", C.c_int32), ("n_surfaces", C.c_int32),
        ("coarse_nv", c_i32p), ("coarse_vx", c_f64p), ("coarse_vy", c_f64p), ("coarse_solid", c_u8p),
        ("fine_off", c_i32p),
        ("cell_nv", c_i32p), ("cell_vx", c_f64p), ("cell_vy", c_f64p), ("cell_mid", c_f64p),
        ("cell_volume", c_f64p), ("cell_surf_id", c_i32p),
        ("kappa", c_f64p), ("sigma_s", c_f64p), ("epsilon", c_f64p), ("uniform_beta", c_f64p),
    ]


class rthx_trace_args(C.Structure):
    _fields_ = [
        ("rays_per_emitter", C.c_int64), ("ray_id_offset", C.c_int64), ("seed", C.c_uint64),
        ("nudge", C.c_double),
        ("n_bins", C.c_int32), ("bins", c_i32p),
        ("mode", C.c_int32), ("locator", C.c_int32),
        ("emitter_rank", C.c_int32), ("emitter_world", C.c_int32),
        ("n_rec_ids", C.c_int32), ("rec_ids", c_i32p), ("rec_bin", C.c_int32),
        ("block_threads", C.c_int32), ("row_chunks", C.c_int32),
    ]


class rthx_rec_out(C.Structure):
    _fields_ = [("capacity", C.c_int64), ("origins", c_f64p), ("endpoints", c_f64p), ("n_recorded", C.c_int64)]


class rthx_stats(C.Structure):
    _fields_ = [
        ("rays_traced", C.c_int64), ("rays_lost", C.c_int64), ("kernel_ms", C.c_double), ("total_ms", C.c_double),
        ("n_blocks", C.c_int32), ("block_threads", C.c_int32), ("row_chunks", C.c_int32), ("smem_bytes", C.c_int32),
        ("hist_in_smem", C.c_int32), ("n_launches", C.c_int32),
    ]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class rthx_smooth_stats(C.Structure):
    _fields_ = [("iterations", C.c_int32), ("launches", C.c_int32), ("delta_init", C.c_double), ("delta", C.c_double),
                ("total_ms", C.c_double), ("ms_per_iteration", C.c_double), ("pass_ms", C.c_double), ("pass_gbs", C.c_double),
                ("dykstra_rounds", C.c_int32), ("pcg_iterations", C.c_int32), ("dykstra_delta", C.c_double),
                ("dykstra_ms", C.c_double), ("converged", C.c_int32), ("pad_", C.c_int32)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class rthx_sparse_stats(C.Structure):
    _fields_ = [("pairs", C.c_int64), ("nnz", C.c_int64), ("flushes", C.c_int64), ("pair_capacity", C.c_int64),
                ("row_groups", C.c_int32), ("hash_slots", C.c_int32), ("reduce_ms", C.c_double)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


RTHX_SMOOTH_FROM_LAST_TRACE, RTHX_SMOOTH_FROM_COUNTS, RTHX_SMOOTH_FROM_F, RTHX_SMOOTH_FROM_CSC = 0, 1, 2, 3
RTHX_SOLVE_FROM_LAST_SMOOTH, RTHX_SOLVE_FROM_DENSE, RTHX_SOLVE_FROM_CSC = 0, 1, 2
RTHX_ROW_MAJOR, RTHX_COL_MAJOR = 0, 1
c_i64p = C.POINTER(C.c_int64)


class rthx_solve_args(C.Structure):
    _fields_ = [("n", C.c_int32), ("source", C.c_int32), ("layout", C.c_int32), ("memory", C.c_int32),
                ("max_iters", C.c_int32), ("measure_pass", C.c_int32),
                ("F_dense", c_f64p), ("colptr", c_i64p), ("rowval", c_i32p), ("nzval", c_f64p),
                ("coeff", c_f64p), ("rhs", c_f64p), ("rtol", C.c_double), ("atol", C.c_double)]


class rthx_solve_stats(C.Structure):
    _fields_ = [("iterations", C.c_int32), ("restarts", C.c_int32), ("launches", C.c_int32), ("converged", C.c_int32),
                ("matvecs", C.c_int32), ("pad_", C.c_int32),
                ("residual", C.c_double), ("rhs_norm", C.c_double), ("total_ms", C.c_double),
                ("matvec_ms", C.c_double), ("matvec_gbs", C.c_double), ("matvec_bytes", C.c_int64)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_ if k != "pad_"}


class rthx_info(C.Structure):
    _fields_ = [
        ("n_elements", C.c_int32), ("n_surfaces", C.c_int32), ("n_cells", C.c_int32), ("n_coarse", C.c_int32),
        ("n_bands", C.c_int32), ("n_affine_faces", C.c_int32), ("device_id", C.c_int32), ("sm_count", C.c_int32),
        ("cc_major", C.c_int32), ("cc_minor", C.c_int32), ("n_bilinear_faces", C.c_int32), ("reserved_", C.c_int32),
    ]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


# every symbol include/rthx.h declares (tests check the built library exports all of them)
EXPORTED_SYMBOLS = (
    "rthx_create", "rthx_create_multi", "rthx_device_count", "rthx_destroy", "rthx_get_info", "rthx_trace_exchange", "rthx_trace_exchange_device",
    "rthx_trace_exchange_multi", "rthx_measure_fp64_peak", "rthx_last_error", "rthx_version",
    "rthx_shared_alloc", "rthx_shared_open", "rthx_shared_close", "rthx_shared_free", "rthx_release_cached",
    "rthx_smooth_F", "rthx_smooth_DkAP", "rthx_solve_grey", "rthx_flag_signal", "rthx_flag_wait", "rthx_host_register", "rthx_host_unregister", "rthx_host_alloc", "rthx_host_free", "rthx_set_copy_helpers", "rthx_counts_nnz", "rthx_counts_csr", "rthx_counts_stats", "rthx_counts_csc",
    "rthx_smooth_sparse", "rthx_smooth_sparse_csc", "rthx_trace_exchange_sparse", "rthx_trace_exchange_continue",
)
