/*
 * rthx.h — C ABI of the B200-native Monte Carlo exchange-factor ray tracer.
 *
 * Drop-in boundary for RayTraceHeatTransfer.jl's `mesh(N_rays; method=:exchange, rec)` path.
 * The reference (pure Julia, no FFI of its own) would bind these entry points with `ccall`
 * from a method that replaces
 *     parallelRayTracing(rtm, rays_total, nudge, verbose; rec)
 *         src/RayTracing/RayTracing2D/ExchangeFactors2D/parallelRayTracing.jl:1-62
 *     computeExchangeFactorsBin(rtm, rays_per_emitter, nudge, spectral_bin, ...)
 *         src/RayTracing/RayTracing2D/ExchangeFactors2D/parallelRayTracing.jl:64-159
 * (see INTEGRATION.md and julia/RTHXExchange.jl).  In this repository the same ABI is driven
 * by the Python `ctypes` twin in raytraceheattransfer.jl_b200/_lib.py.
 *
 * Conventions
 *   - plain C, plain pointers and sizes; the caller owns every host buffer; the library copies the
 *     mesh during rthx_create and never keeps a host pointer after a call returns.
 *   - every function returns an int status: 0 = OK, non-zero = error, message via rthx_last_error.
 *   - indices crossing the ABI are 0-based; -1 = none.
 *   - geometric failures (escaped point location, iteration cap, hit on a non-solid fine wall) are
 *     NOT errors: such rays are dropped and counted in `lost`, exactly like the `nothing` / `-1`
 *     returns of traceRay.jl:37-39,48-50,62-64,69 and getGlobalIndex2D.jl:6.
 *   - there is no CPU fallback: every compute entry point fails with RTHX_ERR_CUDA when no
 *     sm_100 device is usable.
 */
#ifndef RTHX_H
#define RTHX_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RTHX_VERSION_MAJOR 0
#define RTHX_VERSION_MINOR 3

/* status codes */
enum {
  RTHX_OK = 0,
  RTHX_ERR_ARG = 1,      /* bad argument / inconsistent mesh */
  RTHX_ERR_CUDA = 2,     /* CUDA runtime error or no usable device */
  RTHX_ERR_NOMEM = 3,
  RTHX_ERR_INTERNAL = 4
};

/* trace modes.  FIRST_INTERACTION is what method=:exchange computes (traceRay.jl:20-147): every ray
 * stops at its first gas-extinction event or solid-wall hit; albedo and wall reflectivity are applied
 * algebraically later by the unchanged host solver. */
enum {
  RTHX_FIRST_INTERACTION = 0,
  /* Optional total-exchange mode (the analogue of method=:direct's traceSingleRay.jl:7-81 without re-emission; rthx_trace_direct adds it): after
   * every first interaction the ray is absorbed with probability 1 - omega (gas, omega = sigma_s/(kappa+sigma_s)) or
   * epsilon (wall); otherwise it scatters isotropically (isotropicScatter2D.jl:1-4) or is reflected — diffusely about
   * the inward wall normal, or specularly — and is traced on to its next interaction.  counts[i][j] then is the number
   * of rays of emitter i finally ABSORBED by element j.  NOT what method=:exchange feeds to the host solver (that
   * applies albedo and reflectivity algebraically); equals the closure (I - F B)^-1 F (I - B) of the first-interaction
   * F up to discretisation.  Rays still alive after 1000 events face the reference's Russian roulette (:11). */
  RTHX_MULTI_BOUNCE = 1,
  RTHX_MULTI_BOUNCE_SPECULAR = 2
};

/* point-location strategy (rthx_trace_args.locator) */
enum {
  RTHX_LOCATOR_AUTO = 0,     /* analytic lattice inverse on coarse faces verified to be affine sub-meshes,
                                grid + point-in-polygon elsewhere */
  RTHX_LOCATOR_GENERIC = 1   /* uniform grid + crossing-number point-in-polygon everywhere, as
                                findFace2D.jl:1-101 / spatialAccelerations.jl:2-89 */
};

/*
 * Flattened RayTracingDomain2D (DomainStructs.jl:89-130).  One entry per coarse face (user polygon,
 * 3 or 4 CCW vertices) and per fine cell (sub-mesh cell, 3 or 4 CCW vertices), fine cells stored in
 * the walk order of createIndexMapping2D.jl:7-18 (coarse-major, then fine index).
 * Wall i of a polygon spans vertex i -> vertex (i+1) mod nv (PolyVolume2D.jl:8-23).
 * Unused 4th slots of triangles must be present (any value).
 */
typedef struct rthx_mesh {
  int32_t n_coarse;             /* number of coarse faces */
  int32_t n_cells;              /* total number of fine cells  (= Nv) */
  int32_t n_bands;              /* n_spectral_bins (1 for grey) */
  int32_t n_surfaces;           /* Ns = number of solid fine walls */
  const int32_t* coarse_nv;     /* [n_coarse]        3 or 4 */
  const double*  coarse_vx;     /* [n_coarse*4]      vertices */
  const double*  coarse_vy;     /* [n_coarse*4] */
  const uint8_t* coarse_solid;  /* [n_coarse*4]      solidWalls of the coarse face */
  const int32_t* fine_off;      /* [n_coarse+1]      fine cells of coarse c are [fine_off[c], fine_off[c+1]) */
  const int32_t* cell_nv;       /* [n_cells] */
  const double*  cell_vx;       /* [n_cells*4] */
  const double*  cell_vy;       /* [n_cells*4] */
  const double*  cell_mid;      /* [n_cells*2]       midPoint (x,y) */
  const double*  cell_volume;   /* [n_cells]         `volume` field (2-D area) */
  const int32_t* cell_surf_id;  /* [n_cells*4]       global surface index of wall i, -1 if not solid
                                                     (surface_mapping of RayTracingDomain2D.jl:57-76) */
  const double*  kappa;         /* [n_bands*n_cells] kappa_g   */
  const double*  sigma_s;       /* [n_bands*n_cells] sigma_s_g */
  const double*  epsilon;       /* [n_bands*n_surfaces] wall emissivity; may be NULL (only MULTI_BOUNCE
                                                     reads it) */
  const double*  uniform_beta;  /* [n_bands]         uniform_across_bin (validateDomainUniformity.jl:57-85):
                                                     common beta, or -1 when cells disagree */
} rthx_mesh;

/*
 * Arguments of one blocking trace.  Matrix index of an element: surfaces 0..Ns-1 then Ns + cell index
 * (getGlobalIndex2D.jl:5-12).  N = Ns + n_cells.
 *
 * RNG contract (the reference is unseeded; this is new): Philox4x32-10, key = seed,
 * counter = (ray_id lo, ray_id hi, emitter element index, (band << 16) | call#), ray_id in
 * [ray_id_offset, ray_id_offset + rays_per_emitter); two calls per ray, words w0..w3 (call 0), w4..w7 (call 1).
 *   surface emitter: w0 position (32-bit uniform), w1 cos(theta) and w2 psi (23-bit Float32 uniforms, as
 *                    lambertSample2D.jl:2,5 quantises them), (w4,w5) free path (52-bit);
 *   volume emitter : w0 R_1, w1 R_2, w2 triangle selector (quads only), w3 phi (32-bit), (w4,w5) theta (52-bit),
 *                    (w6,w7) free path / optical depth (52-bit).
 *   MULTI_BOUNCE event n (n = 0,1,...): calls 2+2n and 3+2n — decision, azimuth, cos(theta) (walls), roulette (32/23-bit),
 *                    polar angle and next free path (52-bit).
 *   uniforms: (w + 0.5) 2^-32, ((w >> 9) + 0.5) 2^-23, ((hi:lo >> 12) + 0.5) 2^-52 — all in the open interval (0,1).
 * Results are a pure function of
 * (mesh, seed, ray_id range, nudge): independent of thread-block shape, chunking and GPU count.
 */
typedef struct rthx_trace_args {
  int64_t  rays_per_emitter;    /* div(rays_total, N), parallelRayTracing.jl:6 */
  int64_t  ray_id_offset;       /* 0 normally; continuation runs add their counts */
  uint64_t seed;
  double   nudge;               /* 1e4*eps(Float64) by default, multiDispatchRayTrace2D.jl:10 */
  int32_t  n_bins;              /* number of bands traced in this call (batched in the grid) */
  const int32_t* bins;          /* [n_bins] band indices */
  int32_t  mode;                /* RTHX_FIRST_INTERACTION (method=:exchange) | RTHX_MULTI_BOUNCE[_SPECULAR] */
  int32_t  locator;             /* RTHX_LOCATOR_* */
  int32_t  emitter_rank;        /* this call traces emitters e with e % emitter_world == emitter_rank; */
  int32_t  emitter_world;       /*   rows of other emitters are left zero.  (0,1) = all emitters */
  int32_t  n_rec_ids;           /* RayRecorder: number of recorded emitter elements (0 = off) */
  const int32_t* rec_ids;       /* [n_rec_ids] element indices (rec.ids - 1) */
  int32_t  rec_bin;             /* band index whose rays are recorded (rec.bin - 1) */
  int32_t  block_threads;       /* 0 = auto */
  int32_t  row_chunks;          /* thread blocks per (emitter, band) row; 0 = auto */
} rthx_trace_args;

/* RayRecorder output (parallelRayTracing.jl:108,120-123,135-138): origins (post-nudge emission point)
 * and endpoints (interaction point) of every successfully tallied ray of the recorded emitters, in
 * ascending (emitter element, ray id) order.  Caller provides room for `capacity` points each. */
typedef struct rthx_rec_out {
  int64_t  capacity;            /* in points; needs >= n_rec_ids * rays_per_emitter */
  double*  origins;             /* [capacity*2] */
  double*  endpoints;           /* [capacity*2] */
  int64_t  n_recorded;          /* out */
} rthx_rec_out;

typedef struct rthx_stats {
  int64_t rays_traced;          /* rays_per_emitter * owned emitters * n_bins */
  int64_t rays_lost;
  double  kernel_ms;            /* device time of the trace kernel (CUDA events) */
  double  total_ms;             /* device time of the whole call incl. zeroing and copies */
  int32_t n_blocks;
  int32_t block_threads;
  int32_t row_chunks;
  int32_t smem_bytes;
  int32_t hist_in_smem;         /* 1 = per-block shared-memory row histogram, 0 = direct global atomics */
  int32_t n_launches;           /* kernels launched by the call */
} rthx_stats;

typedef struct rthx_info {
  int32_t n_elements;           /* N */
  int32_t n_surfaces;
  int32_t n_cells;
  int32_t n_coarse;
  int32_t n_bands;
  int32_t n_affine_faces;       /* coarse faces whose sub-mesh was verified to be an affine lattice */
  int32_t device_id;
  int32_t sm_count;
  int32_t cc_major, cc_minor;
  int32_t n_bilinear_faces;     /* coarse quadrilaterals that are no parallelograms, verified to be the bilinear lattice of
                                   meshQuad.jl:116-136 (located by the analytic inverse of the bilinear map)          [0.2] */
  int32_t reserved_;
} rthx_info;

typedef struct rthx_handle rthx_handle;

/* Upload the mesh to `device_id`, derive emitter table, edge normals, locator grids, neighbour table and
 * lattice descriptors.  Replaces nothing in the reference (it keeps the mesh in Julia structs); it is the
 * device-side twin of RayTracingDomain2D.jl:2-111 + spatialAccelerations.jl:92-106. */
int rthx_create(rthx_handle** out, const rthx_mesh* mesh, int device_id);
/* The same for n devices at once (one handle each, for rthx_trace_exchange_multi): the host-side derivation runs ONCE, the
 * image is uploaded to all devices concurrently from page-locked memory.  On error no handle is left behind.             [0.3] */
int rthx_create_multi(rthx_handle** out, const rthx_mesh* mesh, const int* device_ids, int n);
int rthx_destroy(rthx_handle* h);
/* Number of usable sm_100 devices (what a `devices = all visible` default of the functor enumerates); RTHX_ERR_CUDA and 0
 * without one.                                                                                                          [0.3] */
int rthx_device_count(int* n);
/* rthx_destroy parks streams, events and device buffers in a per-device pool that the next rthx_create adopts
 * (handles are typically re-created for every trace); this frees everything that is parked. */
int rthx_release_cached(void);
int rthx_get_info(const rthx_handle* h, rthx_info* info);

/* Blocking trace with HOST outputs.  Replaces computeExchangeFactorsBin (parallelRayTracing.jl:64-159)
 * for all `bins` at once: counts_out[b][i][j] = number of rays of emitter i whose first interaction is
 * element j; lost_out[b][i] = rays dropped.  The caller forms F = counts / rowsum exactly as
 * parallelRayTracing.jl:144-146 + row_normalize! :161-169 compose.
 *   counts_out: [n_bins*N*N] uint64 (NULL: leave the counts on the device for rthx_counts_csr / rthx_smooth_F),
 *   lost_out: [n_bins*N] uint64 (may be NULL), rec / stats may be NULL.
 * With emitter_world > 1 only the rows this call owns are written; the other rows of counts_out are NOT touched, so
 * several ranks (processes) can fill one matrix in shared host memory, each copying its rows over its own PCIe link.
 * Pinned / registered destinations are written by DMA directly; pageable ones go through internal pinned staging. */
int rthx_trace_exchange(rthx_handle* h, const rthx_trace_args* args,
                        uint64_t* counts_out, uint64_t* lost_out,
                        rthx_rec_out* rec, rthx_stats* stats);

/* Asynchronous trace into DEVICE buffers on `stream` (a cudaStream_t; NULL = default stream):
 * counts_dev [n_bins*N*N] uint64, lost_dev [n_bins*N] uint64 on the handle's device (or peer-mapped).
 * zero_first: RTHX_ZERO_NONE, RTHX_ZERO_ALL (clear both buffers on the stream before the launch) or
 * RTHX_ZERO_OWN_ROWS (clear only the rows / lost entries of the emitters this call owns — for a matrix shared by
 * several ranks), optionally OR-ed with RTHX_DEST_PEER: the buffers live in ANOTHER device's memory.  A peer-mapped pointer
 * of the same process is recognised by itself; a CUDA-IPC mapping (rthx_shared_open) reports the mapping device, so its
 * callers must say so.  For a peer matrix the chunks of a row add up in a local staging row and the finished row is handed
 * over with plain coalesced stores — no atomics on NVLink, no clearing of the peer rows.                              [0.3]
 * Does not synchronise; stats carries the launch geometry only.  Recording is not available on this entry point. */
enum { RTHX_ZERO_NONE = 0, RTHX_ZERO_ALL = 1, RTHX_ZERO_OWN_ROWS = 2, RTHX_DEST_PEER = 16 };
int rthx_trace_exchange_device(rthx_handle* h, const rthx_trace_args* args,
                               void* counts_dev, void* lost_dev, void* stream,
                               int zero_first, rthx_stats* stats);

/* Single-process multi-GPU trace: emitters are dealt round-robin to the n handles (one per device, same mesh — see
 * rthx_create_multi), one host thread per device drives its launches and copies, all devices run concurrently.
 * args->emitter_rank/world are ignored.
 *   counts_out != NULL: each device copies only the rows it owns into the host matrix, pipelined behind its kernels over its own
 *       PCIe link (rows are disjoint and tile the matrix: no reduction, nothing is cleared on the host);
 *   counts_out == NULL: the devices flush their rows into ONE matrix in the memory of hs[0]'s device through peer access
 *       (NVLink / NVSwitch; finished rows are handed over with plain stores, fused into the trace kernel).  The complete matrix stays resident on
 *       hs[0] for rthx_counts_csr / rthx_counts_csc / rthx_smooth_F / rthx_smooth_DkAP, exactly as after a single-device
 *       rthx_trace_exchange with counts_out == NULL.  Needs peer access between the devices (RTHX_ERR_CUDA otherwise).      [0.3]
 * stats->kernel_ms / total_ms are those of the slowest device. */
int rthx_trace_exchange_multi(rthx_handle** hs, int n, const rthx_trace_args* args,
                              uint64_t* counts_out, uint64_t* lost_out,
                              rthx_rec_out* rec, rthx_stats* stats);

/* Reciprocity smoothing of a dense exchange-factor matrix on the device (next-stage row of the hot path; restates the
 * dense alternating projection of src/HeatTransfer/exchangeFactorSmoothing/smoothExchangeFactors.jl:412-612: build_X,
 * hunger!, scale!, delta_R_X, recover_F).  Returns F_smooth with rows summing to 1 and w_i F_ij = w_j F_ji.
 *   source RTHX_SMOOTH_FROM_LAST_TRACE: the UInt64 counts of traced bin `bin` still resident on the device from the
 *          last rthx_trace_exchange on this handle (no host round trip); n <= N crops to the leading n x n block
 *          (the surfaces-only crop of exchangeRayTracing.jl:9-11);
 *   source RTHX_SMOOTH_FROM_COUNTS / _FROM_F: src_host is a host UInt64 / Float64 [n][n] matrix.
 *   w: [n] reciprocity weights, already renormalised by the caller (smooth_F :452-456); target <= 0 means 8 eps.
 *   measure_pass != 0 additionally times the scaling pass alone (stats->pass_ms / pass_gbs: 16 n^2 bytes per pass). */
enum { RTHX_SMOOTH_FROM_LAST_TRACE = 0, RTHX_SMOOTH_FROM_COUNTS = 1, RTHX_SMOOTH_FROM_F = 2 };
typedef struct rthx_smooth_stats {
  int32_t iterations;
  int32_t launches;
  double  delta_init;           /* delta_R after the first reciprocity projection */
  double  delta;                /* final delta_R */
  double  total_ms;             /* device time: build X + iterations + recover */
  double  ms_per_iteration;
  double  pass_ms;              /* one scaling pass (read + write of X, fused row sums) */
  double  pass_gbs;             /* 16 n^2 bytes / pass_ms */
  int32_t dykstra_rounds;       /* rthx_smooth_DkAP: rounds executed */
  int32_t pcg_iterations;       /* total PCG iterations of the dual solves inside the rounds */
  double  dykstra_delta;        /* delta_perp after the last checked round (delta_perp :DYK, :136-142) */
  double  dykstra_ms;           /* device time of the rounds */
  int32_t converged;            /* 1: delta <= target, or the stalled contraction was accepted below the floor guard
                                   target / sqrt(density) (AP :558-590); 0: max_iters reached — the reference @warns (:605-607) [0.3] */
  int32_t pad_;
} rthx_smooth_stats;
int rthx_smooth_F(rthx_handle* h, int source, const void* src_host, int bin, int n, const double* w, int max_iters,
                  double target, int measure_pass, double* F_out, rthx_smooth_stats* stats);
/* The same with `k_dykstra` Dykstra rounds in front of the alternating projection — DkAP, smoothExchangeFactors.jl:299-318:
 * each round is the orthogonal projection OP (:292-297) onto {reciprocal, unit row sums} through the dual system
 * R lambda = b (Jacobi-PCG, :15-37; the reduced-mass weights Y are formed on the fly, never stored), followed by
 * max(., 0) with the Dykstra correction; the rows are then renormalised and polished by AP.  The reference's own
 * default for a dense F is k_dykstra = 1 when the surface-gas cross-coupling chi >= 0.4, else 0 (:441-450); the caller
 * makes that choice (cross_coupling_chi :215-241 is O(nnz) on the host).  k_dykstra = 0 is rthx_smooth_F. */
int rthx_smooth_DkAP(rthx_handle* h, int source, const void* src_host, int bin, int n, const double* w, int k_dykstra,
                     int max_iters, double target, int measure_pass, double* F_out, rthx_smooth_stats* stats);

/* Reciprocity smoothing of a SPARSE exchange-factor matrix on the device: the sparse branch of smooth_F (density <= 0.25,
 * smoothExchangeFactors.jl:432-434), i.e. AP (:548-612) on the non-zero pattern.  X = (W F + (W F)')/2 is built on the union
 * pattern of F and F' and is exactly symmetric; each iteration is one pass over its non-zeros; the stopping rule is that of
 * rthx_smooth_F.  The result F_smooth keeps that pattern and stays on the device; *nnz_out receives its number of non-zeros and
 * rthx_smooth_sparse_csc copies it out.
 *   source RTHX_SMOOTH_FROM_LAST_TRACE: the UInt64 counts of traced bin `bin` still resident from the last full trace on this
 *          handle (single-device, or rthx_trace_exchange_multi with counts_out == NULL on hs[0]); n <= N crops to the leading
 *          block, row totals are taken over the crop and F_ij = count / row total exactly as rthx_counts_csc computes it;
 *   source RTHX_SMOOTH_FROM_CSC: F given by the host as 0-based CSC, used as given — colptr [n+1] int64, rowval [nnz] int32
 *          strictly ascending within each column, nzval [nnz] float64 (a SparseMatrixCSC, e.g. an F_raw traced in row tiles).
 *          Checked on the host before anything is uploaded: colptr[0] != 0, a decreasing colptr, or a rowval outside [0, n) or
 *          not strictly ascending within its column is RTHX_ERR_ARG.  colptr, rowval and nzval are ignored for FROM_LAST_TRACE.
 * The FROM_CSC result for the F_raw that rthx_counts_csc returns is bit-identical to the FROM_LAST_TRACE result, and
 * repeated calls are bit-identical (fixed summation orders throughout).
 *   w, max_iters, target as for rthx_smooth_F.  stats: the Dykstra fields are 0; measure_pass != 0 times the scaling pass alone,
 *   pass_gbs = (20 nnz_X + 8 (n + 1)) bytes / pass_ms (value read + write, column index, row pointers of X).
 * A sparse smoothing replaces any dense F_smooth on the handle: rthx_solve_grey(RTHX_SOLVE_FROM_LAST_SMOOTH) then fails with
 * RTHX_ERR_ARG until the next rthx_smooth_F; solve a sparse F_smooth with RTHX_SOLVE_FROM_CSC.                            [0.3+] */
enum { RTHX_SMOOTH_FROM_CSC = 3 };
int rthx_smooth_sparse(rthx_handle* h, int source, int bin, int n,
                       const int64_t* colptr, const int32_t* rowval, const double* nzval,
                       const double* w, int max_iters, double target, int measure_pass,
                       int64_t* nnz_out, rthx_smooth_stats* stats);
/* The F_smooth of the last rthx_smooth_sparse on this handle as CSC, with the conventions of rthx_counts_csc: colptr [n+1] int64,
 * rowval [nnz] int64 (rowval_is_i64 != 0) or int32, rows ascending within each column, nzval [nnz]; index_base 0 or 1 is added
 * to colptr and rowval.  RTHX_ERR_ARG when no sparse smoothing has run on the handle.                                     [0.3+] */
int rthx_smooth_sparse_csc(rthx_handle* h, int index_base, int rowval_is_i64,
                           int64_t* colptr, void* rowval, double* nzval);

/* Grey GERT equilibrium solve on the device (next-stage row of the hot path: the consumer of F).  Restates the
 * linear-algebra core of src/HeatTransfer/equilibrium/equilibriumGrey2D.jl:80-211:
 *     M = I - Diagonal(coeff) * F'   (:148-149; coeff = ifelse(Q_known, 1, b), never formed explicitly)
 *     j = M \ h                      (:152-158; restarted GMRES(memory), stop at |r| <= atol + rtol*|h| like
 *                                     Krylov.jl's gmres!(...; memory = 50, restart = true, rtol = 1e-12))
 *     g_i = sum_k F[k,i] j[k]        (:168-194; the caller forms r = b.*g and Abs = (1-b).*g)
 * A caller replaces exactly those lines and keeps populateWorkspace!, the boundary-condition vectors, the
 * temperature recovery and the write-back unchanged on the host.
 *   source RTHX_SOLVE_FROM_LAST_SMOOTH: the n x n F_smooth still resident on the device from the last rthx_smooth_F
 *          on this handle (trace -> smooth -> solve without moving F over PCIe); `n` must match that call;
 *   source RTHX_SOLVE_FROM_DENSE: F_dense is a host [n*n] Float64 matrix, layout RTHX_ROW_MAJOR (C / numpy:
 *          F[i][j] at i*n + j) or RTHX_COL_MAJOR (a Julia `Matrix` as it lies in memory);
 *   source RTHX_SOLVE_FROM_CSC: colptr [n+1] / rowval [nnz] / nzval [nnz], the fields of a SparseMatrixCSC, 0-based.
 *   coeff, rhs: [n].  memory <= 0 -> 50; max_iters <= 0 -> 2n (Krylov.jl's itmax); rtol <= 0 -> 1e-12;
 *   atol < 0 -> sqrt(eps) (Krylov.jl's default).  j_out [n]; g_out [n] may be NULL.
 *   measure_pass != 0 additionally times the product y = F'x alone (stats->matvec_ms / matvec_gbs). */
enum { RTHX_SOLVE_FROM_LAST_SMOOTH = 0, RTHX_SOLVE_FROM_DENSE = 1, RTHX_SOLVE_FROM_CSC = 2 };
enum { RTHX_ROW_MAJOR = 0, RTHX_COL_MAJOR = 1 };
typedef struct rthx_solve_args {
  int32_t n;
  int32_t source;               /* RTHX_SOLVE_FROM_* */
  int32_t layout;               /* FROM_DENSE: RTHX_ROW_MAJOR | RTHX_COL_MAJOR */
  int32_t memory;               /* Krylov subspace cap per restart cycle */
  int32_t max_iters;            /* cap on the total number of inner iterations */
  int32_t measure_pass;
  const double*  F_dense;       /* FROM_DENSE */
  const int64_t* colptr;        /* FROM_CSC */
  const int32_t* rowval;
  const double*  nzval;
  const double*  coeff;         /* [n] */
  const double*  rhs;           /* [n] h */
  double rtol;
  double atol;
} rthx_solve_args;
typedef struct rthx_solve_stats {
  int32_t iterations;           /* inner (Arnoldi) iterations */
  int32_t restarts;
  int32_t launches;
  int32_t converged;            /* 1: true residual |h - M j| <= atol + rtol*|h| */
  int32_t matvecs;              /* products with F' (one read of F each) */
  int32_t pad_;
  double  residual;             /* final true residual norm */
  double  rhs_norm;
  double  total_ms;             /* device time of the whole solve */
  double  matvec_ms;            /* one product y = F'x (measure_pass) */
  double  matvec_gbs;           /* matvec_bytes / matvec_ms */
  int64_t matvec_bytes;         /* algorithmic bytes of one product: 8 n^2 (dense) or 12 nnz + 8 (n+1) (CSC) */
} rthx_solve_stats;
int rthx_solve_grey(rthx_handle* h, const rthx_solve_args* args, double* j_out, double* g_out, rthx_solve_stats* stats);

/* Sparse (CSR) read-out of the counts still resident on the device from the last rthx_trace_exchange on this handle
 * (all emitters): per row the non-zero absorber columns in ascending order — exactly the triplets the reference
 * feeds to sparse(I, J, V) (parallelRayTracing.jl:144-154) — compacted on the device, so optically thick meshes
 * (test/test_2d_diffusion.jl:64) never move their N^2 zeros.  rthx_trace_exchange accepts counts_out == NULL for
 * callers that only want this view.
 *   rthx_counts_nnz : number of non-zeros of traced bin `bin` (also prepares the row pointers on the device);
 *   rthx_counts_csr : row_ptr [R+1], cols [nnz], vals [nnz] (may be NULL), F_vals [nnz] = count / row total (may be
 *                     NULL; this is the row-normalised F of row_normalize!, :161-169), row_lost not included.
 * R = N after a trace of all emitters.  After a SHARDED trace (emitter_world > 1) the resident rows are those the call owned,
 * R = ceil((N - emitter_rank) / emitter_world), row y being element emitter_rank + y * emitter_world: meshes whose dense
 * 8 N^2-byte matrix does not fit (N >> 57 k elements) are traced as a sequence of such row tiles on one device, each read out
 * as CSR and merged on the host (raytraceheattransfer.jl_b200/_lib.py trace_row_tiles).                               [0.3] */
int rthx_counts_nnz(rthx_handle* h, int bin, int64_t* nnz_out);
int rthx_counts_csr(rthx_handle* h, int bin, int64_t* row_ptr, int32_t* cols, uint64_t* vals, double* F_vals);
/* The same counts as the three arrays of a compressed-sparse-COLUMN matrix — the memory layout of the SparseMatrixCSC{Float64,Int}
 * that computeExchangeFactorsBin returns (parallelRayTracing.jl:154-158), so the caller wraps them and neither runs
 * sparse(I, J, V) over ~1e8 triplets nor transposes a CSR matrix on the host:
 *   colptr [N+1] int64, rowval [nnz] int64 (rowval_is_i64 != 0; Julia `Int`) or int32 (scipy), rows ascending within a column,
 *   vals [nnz] counts (may be NULL), F_vals [nnz] = count / row total (may be NULL);
 *   index_base 0 or 1 is added to colptr and rowval (1 = Julia).
 * rthx_counts_stats: non-zeros of the bin and the surface-gas cross-coupling chi of its row-normalised F
 *   (cross_coupling_chi, smoothExchangeFactors.jl:212-241: sum of F_ij with exactly one of i, j a surface, over N) — what
 *   smooth_F needs to choose its branch (:421-450) without touching the matrix on the host.                               [0.3] */
int rthx_counts_stats(rthx_handle* h, int bin, int64_t* nnz_out, double* chi_out);
int rthx_counts_csc(rthx_handle* h, int bin, int index_base, int rowval_is_i64, int64_t* colptr, void* rowval, uint64_t* vals, double* F_vals);

/* Blocking trace whose counts never exist in dense form: a hashed row tally for meshes whose 8 N^2-byte count matrix does not fit
 * (N >> 57 k elements).  Each thread block tallies its row in a shared-memory hash table and flushes it as (row, column, count)
 * pairs into a pair buffer; the pairs are radix-sorted and reduced by key into u64 totals that stay on the device.  Device memory
 * is O(non-zeros), not O(rows x N).  The pair buffer holds at most half the free device memory; a group of rows whose pairs
 * overrun it is traced again split in two (exact: counts are a pure function of seed, ray id and emitter).
 * Same arguments, lost_out, rec and stats as rthx_trace_exchange with counts_out == NULL; sharded traces (emitter_rank/world),
 * ray_id_offset, batched bins, both locators and the recorder work as there.  RTHX_MULTI_BOUNCE[_SPECULAR] is RTHX_ERR_ARG.
 * Afterwards rthx_counts_nnz / _csr / _stats / _csc and rthx_smooth_sparse(RTHX_SMOOTH_FROM_LAST_TRACE) return what they return
 * after rthx_trace_exchange(counts_out == NULL) with the same arguments, bit for bit; rthx_smooth_F / rthx_smooth_DkAP
 * (RTHX_SMOOTH_FROM_LAST_TRACE) fail with RTHX_ERR_ARG until the next dense trace, which in turn discards the sparse form.
 * sparse_stats (may be NULL) reports the tally.                                                                           [0.3+] */
typedef struct rthx_sparse_stats {
  int64_t pairs;                /* pairs flushed by the launches that completed */
  int64_t nnz;                  /* non-zeros of all traced bins after the reduction */
  int64_t flushes;              /* hash-table flushes of those launches (one per block at least) */
  int64_t pair_capacity;        /* pair-buffer capacity in pairs */
  int32_t row_groups;           /* launches that completed: 1 + the number of splits after an overflow */
  int32_t hash_slots;           /* hash-table slots per block */
  double  reduce_ms;            /* device time of sort + reduce-by-key */
} rthx_sparse_stats;
int rthx_trace_exchange_sparse(rthx_handle* h, const rthx_trace_args* args, uint64_t* lost_out, rthx_rec_out* rec, rthx_stats* stats,
                               rthx_sparse_stats* sparse_stats);

/* Continue the trace whose counts are resident: add the rays [ray_id_offset, ray_id_offset + rays_per_emitter) of every owned emitter
 * to them, in the form they are in (dense or hashed).  The resident counts are always those of ONE trace of a contiguous ray-id range
 * [lo, hi) with one seed, so k continuations give, bit for bit, what one trace of the whole range gives: rthx_counts_nnz / _csr / _stats
 * / _csc, rthx_smooth_sparse(RTHX_SMOOTH_FROM_LAST_TRACE) and, for the dense form, rthx_smooth_F / _DkAP(RTHX_SMOOTH_FROM_LAST_TRACE).
 * Preconditions (RTHX_ERR_ARG naming the mismatch, the resident state untouched): counts are resident from rthx_trace_exchange with
 * counts_out == NULL or from rthx_trace_exchange_sparse (not from a host-output trace, nor from rthx_trace_exchange_multi, whose peer
 * hand-over stores rows instead of adding them); seed, nudge, mode, locator, bins (in the same order) and emitter_rank / emitter_world
 * are those of that trace; ray_id_offset == hi.  rays_per_emitter, block_threads and row_chunks are free: counts do not depend on the
 * launch shape.  Afterwards hi has advanced by rays_per_emitter.
 *   dense form : the launches of rthx_trace_exchange(counts_out == NULL) without clearing the counts (MULTI_BOUNCE too);
 *   hashed form: the new rays are tallied and reduced into a sorted set of their own (row groups and splits as rthx_trace_exchange_sparse),
 *                which a merge-path kernel merges into the resident set, summing equal keys; the merged set then replaces it.
 *                Device memory at its peak, 16 bytes a key: while the new rays are tallied, the resident set, the pair buffer (24 bytes a
 *                pair, as rthx_trace_exchange_sparse sizes it) and the new set (up to 2.5x it while it grows: the old and the grown copy);
 *                during the merge, the resident, the new and the merged set (old nnz + new nnz), with the pair buffer released first
 *                when the merged set would not fit beside it.  The old and the new set are freed after the merge.
 * lost_out [n_bins*N] (may be NULL) and stats->rays_lost are cumulative over [lo, hi); stats->rays_traced and the kernel times are this
 * call's.  The recorder records this call's rays only, as a plain trace with this ray_id_offset would.  sparse_stats (may be NULL;
 * zeroed for the dense form): this call's pairs, flushes and row groups, nnz after the merge, reduce_ms including the merge.
 * The prepared row / column pointers of the read-outs are rebuilt on the next read-out; an F_smooth left on the device by an earlier
 * rthx_smooth_F / rthx_smooth_sparse is NOT updated (smooth again).  A call that fails after its checks leaves no counts resident, with
 * one exception: a hashed continuation that fails before its merged set is complete (e.g. RTHX_ERR_NOMEM, RTHX_ERR_CUDA from an
 * allocation) leaves the resident set and its lost counters as they were.                                               [0.3+] */
int rthx_trace_exchange_continue(rthx_handle* h, const rthx_trace_args* args, uint64_t* lost_out, rthx_rec_out* rec, rthx_stats* stats,
                                 rthx_sparse_stats* sparse_stats);

/* Blocking trace of the emitter rows a caller names, and no others: what the surfaces-only crop of exchangeRayTracing.jl:9-11 keeps
 * (emitters = 0..Ns-1 of a transparent enclosure, where the other Nv rows would be traced and thrown away), or the exchange factors
 * of a few elements (one heater, one sensor).  Row y is element emitters[y]; its counts are those of the same row of a full
 * rthx_trace_exchange with the same args, bit for bit (the RNG contract keys every ray by seed, ray id, emitter and band), and
 * rays_per_emitter is that of the full trace (div(rays_total, N), not div(rays_total, R)).
 *   emitters [n_emitters]: R = n_emitters >= 1 element indices, strictly ascending, in [0, N).  args as for rthx_trace_exchange (seed,
 *       bins, mode incl. both MULTI_BOUNCE modes, locator, ray_id_offset, launch shape), except that emitter_rank / emitter_world must be
 *       (0, 1) and rec_ids must be a subset of the list.  A violation is RTHX_ERR_ARG naming it, with nothing resident changed; a list
 *       whose 8 R N n_bins bytes of counts do not fit in device memory is RTHX_ERR_NOMEM (split the list).
 *   counts_out: [n_bins][R][N] uint64, row y = element emitters[y] (NULL: leave the R rows resident on the device);
 *   lost_out:   [n_bins][N] uint64 (may be NULL), 0 for unlisted elements;  stats->rays_traced = rays_per_emitter * R * n_bins.
 * Read-outs of the resident rows afterwards (each equal, bit for bit, to the same call after the full trace restricted to the listed rows):
 *   rthx_counts_nnz / _csr : the R listed rows, as after a sharded trace;
 *   rthx_counts_stats / _csc: the N x N matrix whose unlisted rows are empty (nnz and chi over the listed rows);
 *   rthx_smooth_F / _DkAP / rthx_smooth_sparse (RTHX_SMOOTH_FROM_LAST_TRACE) with crop n: accepted when every row < n is listed, else
 *       RTHX_ERR_ARG naming the first missing row.
 * rthx_trace_exchange_continue after a resident rows trace continues the same list (the handle keeps it).                [0.3+] */
int rthx_trace_exchange_rows(rthx_handle* h, const rthx_trace_args* args, const int32_t* emitters, int32_t n_emitters,
                             uint64_t* counts_out, uint64_t* lost_out, rthx_rec_out* rec, rthx_stats* stats);

/* method=:direct of the reference's functor, grey: energy bundles traced to absorption, re-emitted by every element whose temperature is
 * unknown.  Source y is element sources[y] and traces rays[y] bundles (ray ids [ray_id_offset, ray_id_offset + rays[y])) with the events
 * of RTHX_MULTI_BOUNCE[_SPECULAR] (args->mode).  A bundle absorbed by element k is tallied in row y, column k; if reemit[k] != 0 it then
 * leaves k again as a fresh emission of k (uniform point, Lambert about the inward normal / isotropic, emission nudge, new free path) and
 * goes on, else it ends.  Re-emission m of a bundle draws Philox calls 0x8000 + 2m and 0x8001 + 2m (counter word 2 stays the source), so
 * with no absorption at a re-emitting element the counts are, bit for bit, those of rthx_trace_exchange_rows(sources) with the same mode.
 * The event counter runs over the whole chain: roulette after 1000 events also ends chains in an enclosure without a sink.
 *   sources [n_sources]: strictly ascending element indices; rays [n_sources] >= 1; reemit [N] flags; bundle_energy [n_sources] >= 0;
 *   absorbed_out [N]: Abs_k = sum_y bundle_energy[y] count[y][k], summed on the device in ascending y with every product and sum
 *       rounded on its own — bit-identical for any launch shape, and to the same sum over rows read out with rthx_counts_csr;
 *   lost_out [N] (may be NULL): bundles of source element e lost (escaped, roulette, 16000 events); events_out (may be NULL): traversal
 *       segments of all bundles (one per interaction or loss); stats (may be NULL): rays_traced = sum of rays.
 * args: n_bins = 1, n_rec_ids = 0, emitter_rank / emitter_world (0, 1); seed, nudge, locator, ray_id_offset, block_threads and
 * row_chunks as for a trace.  A violation is RTHX_ERR_ARG naming it, with nothing resident changed.  Afterwards the counts of the
 * sources stay resident as the listed rows of a rows trace: rthx_counts_nnz / _csr / _stats / _csc read them;
 * rthx_trace_exchange_continue and the smoothings refuse them.                                                          [0.3+] */
int rthx_trace_direct(rthx_handle* h, const rthx_trace_args* args, const int32_t* sources, const int64_t* rays, int32_t n_sources,
                      const uint8_t* reemit, const double* bundle_energy, double* absorbed_out, uint64_t* lost_out, int64_t* events_out,
                      rthx_stats* stats);

/* rthx_trace_direct with the redirection tally, for the radiosity, irradiation and intensity fields.  A redirection is an event at
 * element k that neither ends nor re-emits the bundle: a scattering in cell k (dec < omega_k) or a reflection at surface k
 * (dec >= eps_k).  Each one is tallied in row y, column k of a second count block, from the decision already drawn (no new Philox
 * draw), so the absorption counts, absorbed_out, lost_out and events_out are bit for bit those of rthx_trace_direct with the same
 * arguments, and events = sum of absorption counts + sum of redirection counts + sum of lost.
 *   redirected_out [N] (not NULL): r_k = sum_y bundle_energy[y] redir[y][k], the fixed-order sum of absorbed_out over the second block.
 * Arguments and checks otherwise those of rthx_trace_direct.  The two blocks take 16 R N bytes of device memory; if they cannot fit the
 * call is RTHX_ERR_NOMEM naming the bytes, with nothing resident changed.  Afterwards the resident record holds two bins: bin 0 the
 * absorption counts, bin 1 the redirection counts, both read by rthx_counts_nnz / _csr / _stats / _csc (after rthx_trace_direct, bin 1
 * is RTHX_ERR_ARG); rthx_trace_exchange_continue and the smoothings refuse them.                                        [0.3+] */
int rthx_trace_direct_fields(rthx_handle* h, const rthx_trace_args* args, const int32_t* sources, const int64_t* rays, int32_t n_sources,
                             const uint8_t* reemit, const double* bundle_energy, double* absorbed_out, double* redirected_out,
                             uint64_t* lost_out, int64_t* events_out, rthx_stats* stats);

/* rthx_trace_direct (redirected_out == NULL) or rthx_trace_direct_fields (redirected_out != NULL) on the hashed row tally of
 * rthx_trace_exchange_sparse, for source lists whose 8 R N bytes of dense counts (16 R N with the redirection tally) do not fit: an
 * isothermal or prescribed-temperature medium makes every element a source, R = N.  Each block tallies its source row in a
 * shared-memory hash table; the table is flushed between rounds of bundles once it is half full, and inside a round a tally that finds
 * neither its key nor an empty slot within a fixed probe length is appended to the pair buffer as its own (key, 1) pair (a bundle
 * tallies at every absorption by a re-emitting element and every redirection, with no block-wide point to flush at).  The pairs are
 * sorted and reduced by key, so the totals do not depend on where a tally landed.  Row y's absorptions are row key y * blocks, its
 * redirections y * blocks + 1 (blocks = 1, or 2 with the redirection tally).  The pair buffer takes at most half the free device
 * memory; a group of source rows whose pairs overrun it is traced again split in two, and one source row that overruns it alone is
 * RTHX_ERR_NOMEM naming the source, with nothing resident (as rthx_trace_exchange_sparse).
 *   absorbed_out / redirected_out: the sums of rthx_trace_direct(_fields), bit for bit: the sorted set is transposed to columns and
 *       each column summed in ascending source row, with every product and sum rounded on its own (a zero count adds +0.0);
 *   lost_out, events_out, stats: as rthx_trace_direct, counted once however often a group was traced; sparse_stats (may be NULL):
 *       the tally, as rthx_trace_exchange_sparse reports it.
 * Arguments and checks are those of rthx_trace_direct(_fields) without the check of the dense counts against free memory.  Afterwards
 * rthx_counts_nnz / _csr / _stats / _csc for bins 0 (and 1) return what they return after rthx_trace_direct(_fields) with the same
 * arguments, bit for bit; rthx_trace_exchange_continue and the smoothings refuse the counts.  A set of more than 2^31 - 1
 * non-zeros in one count block cannot be summed (RTHX_ERR_ARG naming the limit).                                       [0.3+] */
int rthx_trace_direct_sparse(rthx_handle* h, const rthx_trace_args* args, const int32_t* sources, const int64_t* rays, int32_t n_sources,
                             const uint8_t* reemit, const double* bundle_energy, double* absorbed_out, double* redirected_out,
                             uint64_t* lost_out, int64_t* events_out, rthx_stats* stats, rthx_sparse_stats* sparse_stats);

/* Peer-memory plumbing for the fused flush in one-process-per-GPU runs: rank 0 allocates the UInt64 count matrix
 * with rthx_shared_alloc and publishes the 64-byte CUDA IPC handle; every other rank maps it with rthx_shared_open
 * (peer access over NVLink is enabled lazily) and passes the mapped pointer as `counts_dev` to
 * rthx_trace_exchange_device with zero_first = RTHX_ZERO_OWN_ROWS | RTHX_DEST_PEER (an IPC mapping reports the mapping device: the caller
 * declares it).  Each rank's kernel then hands its own (disjoint) finished rows over to rank 0's memory with plain coalesced
 * stores over NVLink — the "reduce" is fused into the trace kernel, nothing on the wire is atomic and only the step flags
 * below remain. */
int rthx_shared_alloc(int device_id, uint64_t bytes, void** dev_ptr, unsigned char ipc_handle[64]);
int rthx_shared_open(int device_id, const unsigned char ipc_handle[64], void** dev_ptr);
int rthx_shared_close(int device_id, void* dev_ptr);
int rthx_shared_free(int device_id, void* dev_ptr);

/* Step flags for the fused flush without a host-launched collective per step: 64-bit counters in the matrix owner's memory.
 * rthx_flag_signal enqueues a system-scope release store of `value` to *flag (device memory, possibly peer-mapped) behind
 * everything already on `stream` — a rank signals "my rows of step s have landed" after its trace kernel; rthx_flag_wait
 * enqueues an acquire spin until flags[0..n) >= value in front of whatever follows on `stream`.  A wait gives up after
 * timeout_s (<= 0: 30 s) and increments *err_flag (may be NULL) so that a dead peer cannot hang the device.                [0.3] */
int rthx_flag_signal(void* flag, uint64_t value, void* stream);
int rthx_flag_wait(const void* flags, int n, uint64_t value, double timeout_s, void* err_flag, void* stream);

/* Page-lock a caller-owned host buffer (e.g. a matrix in POSIX shared memory that several ranks fill) so the
 * pipelined device->host copies of rthx_trace_exchange run at full PCIe speed and overlap with tracing. */
int rthx_host_register(void* ptr, uint64_t bytes);
int rthx_host_unregister(void* ptr);
/* After a multi-GPU trace the result arrays (CSC arrays, F_smooth: ~1 GB each for cfg3) live on ONE device and their device->host
 * copies are bound by that device's PCIe link while the other links idle.  rthx_set_copy_helpers registers the handles on the other
 * devices: large copies into page-locked memory are then cut into one slice per device, each slice hopping to its helper over
 * NVLink and leaving through that device's own link.  n = 0 clears the list; the helpers must outlive their use.          [0.3] */
int rthx_set_copy_helpers(rthx_handle* h, rthx_handle** helpers, int n);

/* Page-locked host memory for output arrays (count matrix, CSC arrays, F_smooth): device->host copies into it run by DMA at
 * full PCIe speed with no staging pass.  A Julia caller wraps the pointer with unsafe_wrap(Array, ptr, dims).            [0.3] */
int rthx_host_alloc(void** ptr, uint64_t bytes);
int rthx_host_free(void* ptr);

/* FP64 FMA-chain micro-benchmark on the handle's device: the denominator of the FP64 roofline
 * (MEASURED_PEAKS.json has no FP64 entry).  Returns TFLOP/s (2 flop per DFMA). */
int rthx_measure_fp64_peak(rthx_handle* h, double* tflops);

/* Message of the last error on this handle (h == NULL: last error of rthx_create on this thread). */
const char* rthx_last_error(const rthx_handle* h);
int rthx_version(void);

#ifdef __cplusplus
}
#endif
#endif /* RTHX_H */
