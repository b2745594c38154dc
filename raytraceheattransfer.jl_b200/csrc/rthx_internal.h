// rthx_internal.h — structures shared between the host API (rthx_api.cu) and the kernels (rthx_kernels.cu).
#pragma once
#include <cstddef>
#include <cstdint>
#include <cuda_runtime.h>

#include "rthx.h"

namespace rthx {

enum : int { KIND_GENERIC = 0, KIND_AFFINE_QUAD = 1, KIND_AFFINE_TRI = 2, KIND_BILINEAR_QUAD = 3 };

constexpr int LOGTAB_N = 256;   // entries of the -log table staged in shared memory by every block (csrc/rthx_logtab.h, 16 bytes each)

// One coarse face (user polygon).  Staged in shared memory by every thread block when the whole array fits.
struct alignas(16) CoarseDev {
  double vx[4], vy[4];   // CCW vertices
  double nx[4], ny[4];   // unit outward edge normals (the reference's `inwardNormals`, calculateInwardNormal.jl:1-12)
  double h[4];           // plane offsets: quads h0 = v0·n0, h1 = v1·n1, h2 = v2·n0, h3 = v3·n1 (slab form); else h_i = v_i·n_i
  double cen[2], hw[2];  // quads: centre line (h_a + h_{a+2})/2 and half width (h_a - h_{a+2})/2 of the edge pair with normal n_a
  // affine lattice inverse (kinds 1,2): s = (p-a)·g1, t = (p-a)·g2, lattice cell (floor s, floor t) in [0,Nx)x[0,Ny)
  // bilinear lattice (kind 3, a convex quadrilateral that is no parallelogram: meshQuad.jl:116-136 maps the unit square by
  //   P(s,t) = A + s E + t F + s t G): a = A, g1 = E = B-A, g2 = F = D-A, cen = G = A-B+C-D, hw[0] = 1/(E x G), hw[1] unused;
  //   h_i = v_i·n_i for all four edges (no slab form)
  double ax, ay, g1x, g1y, g2x, g2y;
  int32_t nv;
  int32_t kind;
  int32_t Nx, Ny;
  int32_t fine_off;      // first fine cell (global cell index)
  int32_t lat_off;       // kind 2: offset of this face's lattice -> local fine index table, else -1
  int32_t diag;          // kind 2: 0-based coarse edge that is the cut diagonal, else -1
  int32_t nbr[4];        // coarse face across edge k (-1: locate generically / none)
  uint8_t solid[4];
  int32_t abs_off;       // kinds 1,2: first row of this face in the absorber table (5 entries per lattice cell), else -1
};
static_assert(sizeof(CoarseDev) % 16 == 0, "CoarseDev must stay a multiple of 16 bytes (shared-memory layout behind it)");

// Uniform-grid face set for the reference-faithful locator (spatialAccelerations.jl:2-59).
// Set 0 = coarse mesh, set 1+c = fine cells of coarse face c.
struct FaceSetDev {
  double ox, oy;         // grid origin
  double inv_cx, inv_cy; // 1 / bucket size per axis
  int32_t nx, ny;
  int32_t bucket_off;    // first bucket of this set in bucket_ent
  int32_t poly_base;     // local face f of this set is polygon poly_base + f (cells first, then coarse faces)
};
static_assert(sizeof(FaceSetDev) == 48, "FaceSetDev is read with three 16-byte loads");

struct TraceParams {
  // mesh (device pointers)
  const CoarseDev* coarse;
  const FaceSetDev* sets;
  const int4* bucket_ent;      // per bucket {code, a, b, c}: -1 empty | 0 sole face a | k = 1..3 candidates a, b, c | k > 3 candidates bucket_cand[a .. a+k)
  const int32_t* bucket_cand;
  const double* face_rec;      // [n_poly*12] one 96-byte record per polygon: vx[4], vy[4] (a triangle repeats vertex 0 in slot 3), {vertex count,
                               // normal-orientation bits, surface ids of walls 0..3} (rthx_api.cu, face_record)
  const int32_t* poly_nv;
  const double* poly_vx;       // [n_poly*4]
  const double* poly_vy;
  const double* poly_nx;       // [n_cells*4] unit outward normals per cell edge (generic tables only)
  const double* poly_ny;
  const double* cell_mid;      // [n_cells*2]
  const double* cell_volume;   // [n_cells]
  const int32_t* cell_surf_id; // [n_cells*4]
  const double* beta;          // [n_bands*n_cells]
  const double* uniform_beta;  // [n_bands]
  const double* omega;         // [n_bands*n_cells]    scattering albedo sigma_s/(kappa+sigma_s)   (MULTI_BOUNCE)
  const double* band_u;        // [n_bands*2] {albedo shared by every cell, emissivity shared by every surface} of the band, -1 where they differ
                               // (the MULTI queue kernel then skips the per-cell / per-surface load)
  const double* eps;           // [n_bands*n_surfaces] wall emissivity                              (MULTI_BOUNCE)
  const int32_t* lattice;      // lattice -> local fine index tables (kind 2)
  const int32_t* abs_tab;      // affine faces: [lattice cell][gas | wall on coarse edge 0..3] -> absorber index or -1
  const int32_t* em_cell;      // [N]
  const int32_t* em_wall;      // [N]  -1 for volume emitters
  const int32_t* em_coarse;    // [N]
  const int32_t* bins;         // [n_bins] traced band indices
  const int32_t* rec_slot;     // [N] recorder slot of element or -1 (nullptr = recording off)
  // outputs
  unsigned long long* counts;  // row (bi, y) at ((bi*rows_per_bin + y) * N)
  unsigned long long* lost;    // [n_bins*N]
  unsigned long long* peer_counts;  // fused multi-GPU flush: the matrix in peer memory ([n_bins][N][N]) that finished rows are handed
                                    // over to; `counts` is then a local compact staging matrix.  nullptr: `counts` is the destination
  unsigned int* row_done;      // [n_bins*n_owned] chunks of a row that have flushed (hand-over ticket), with peer_counts
  double* rec_pts;             // [n_rec*rays_per_emitter*4] origin xy, endpoint xy
  uint8_t* rec_valid;          // [n_rec*rays_per_emitter]
  // scalars
  int32_t n_coarse, n_cells, n_surfaces, N;
  int32_t n_bins;
  int32_t emitter_rank, emitter_world, n_owned;
  int32_t y_offset;            // first owned-emitter ordinal of this launch (row batches for copy/compute overlap)
  int32_t compact_rows;        // 1: counts row index is the owned-emitter ordinal, 0: the element index
  int32_t row_chunks;
  int32_t coarse_in_smem;
  int32_t force_generic;
  int32_t specular;            // MULTI_BOUNCE: mirror reflection instead of diffuse
  int32_t flush_system;        // 1: system-scope atomics for the flush (count matrix in peer memory)
  int32_t rec_bin;
  int32_t queue_refill;        // queue kernel: with the queue dry, emit the next batch once <= this many lanes still hold a ray
  int32_t queue_sq;            // MULTI queue kernel: the domain is one parallelogram (1 axis-aligned, 2 general): SQ form of the step
  // The 64-bit block below starts on a 16-byte boundary of the parameter bank whatever the number of pointers above: the kernels take
  // the constants and the Philox round keys as c[0][..] operands / 128-bit uniform loads, and ptxas' register allocation depends on
  // their alignment.  Measured when a pointer was dropped above (everything slid by 8 bytes, rk[] to an address = 8 mod 16): the
  // MULTI_BOUNCE queue kernel went from 127 to 377 local-memory instructions (stack 64 -> 88 bytes) and from 3.48e10 to 2.97e10 rays/s
  // on cfg3 (profiles/r4/r4c_*), the SQ kernel from 3 to 9.
  alignas(16) int64_t rays_per_emitter;
  int64_t ray_id_offset;
  uint64_t seed;
  double nudge;
  // constants kept in the parameter bank so FP64 instructions can take them as c[0][..] operands
  double k_u52;   // 1 - 2^-53
  double k_u32;   // 1 - 2^-33
  double k_eps;   // 1e-10, the near-parallel threshold of distToSurface2D.jl:10
  double k_u52c;  // 3/2 - 2^-53: mantissa injection minus this = uniform - 1/2
  double k_u32c;  // 3/2 - 2^-33
  // SQ kernels (single parallelogram face): slab centre lines / half widths, folded lattice offsets, axis-aligned special case
  double sq_cen0, sq_hw0, sq_cen1, sq_hw1;
  double sq_lc1, sq_lc2, sq_one_m_nudge;
  double sq_cy, sq_cx;         // axis-aligned: n0y * cen0, n1x * cen1
  uint32_t sq_flip0, sq_flip1; // axis-aligned: sign bit of n0y / n1x
  int32_t sq_axis;
  int32_t sq_pad_;
  uint32_t rk[20];  // Philox round keys (key + r*W), two per round
  CoarseDev face0;  // SQ kernels: the single coarse face, read from the parameter bank
  // Hashed row tally (rthx_trace_exchange_sparse).  Kept behind everything else so that no field the other kernels read moves.
  unsigned long long* sk_keys; // [sk_cap] pair keys (row key << 32) | column, row key = y * n_bins + bi; nullptr: no hashed tally
  uint32_t* sk_cnt;            // [sk_cap] pair counts
  unsigned long long* sk_ctl;  // [0] pairs reserved, [1] overflow flag, [2] flushes
  unsigned long long sk_cap;   // pair-buffer capacity
  int32_t sk_slots_log2;       // hash slots per block = 1 << sk_slots_log2 (>= 2 blockDim.x)
  int32_t sk_pad_;
  // method=:direct (rthx_trace_direct), behind everything else as well
  const int64_t* dr_rays;      // [listed rows] bundles of source row y
  const uint8_t* dr_reemit;    // [N] 1: the element's temperature is unknown, a bundle it absorbs is emitted again from it
  unsigned long long* dr_events;  // [1] traversal segments of all bundles (one per interaction, or per loss)
  // method=:direct with the redirection tally (rthx_trace_direct_fields), behind the fields above
  int32_t dr_redirect;         // 1: every scattering / reflection at element k is tallied in row y, column k of the second count block
                               // (rows n_owned + y: the compact layout of a two-bin rows trace)
  int32_t dr_pad_;
};

static_assert(offsetof(TraceParams, rays_per_emitter) % 16 == 0 && offsetof(TraceParams, k_u52) % 16 == 0 && offsetof(TraceParams, rk) % 16 == 0,
              "TraceParams: constants and round keys keep their 16-byte alignment in the parameter bank");

// Which trace kernel runs: decided once per trace by make_plan (rthx_api.cu), mapped to its compiled instance by rthx_kernels.cu.
struct TraceKernelSel {
  enum Family : int {
    LOCKSTEP,   // trace_exchange_kernel: one ray per thread, any mesh
    SQ,         // trace_exchange_sq_kernel: the whole domain is one parallelogram face
    QUEUE,      // trace_exchange_queue_kernel: per-warp ray queue (multi-face meshes; MULTI_BOUNCE on analytic meshes)
    HASH,       // trace_exchange_hash_kernel: hashed row tally (rthx_trace_exchange_sparse)
    DIRECT,     // trace_direct_kernel: MULTI_BOUNCE with re-emission (rthx_trace_direct)
    DIRECT_HASH,  // trace_direct_hash_kernel: the same with the hashed row tally (rthx_trace_direct_sparse)
  };
  Family family = LOCKSTEP;
  bool hist = false;      // row histogram in shared memory (SQ and QUEUE always, HASH never)
  bool fast = false;      // no generic locator in the kernel: every face an affine lattice with a complete neighbour table.  The
                          // generic locator tables (ensure_generic) are needed exactly when this is false.
  bool multi = false;     // MULTI_BOUNCE event loop
  int depth = 0;          // QUEUE: rays parked per lane and batch (queue slots per warp = 32 * depth)
  bool general = false;   // QUEUE: bilinear lattices or interfaces without a unique neighbour (the !fast build has them always)
  bool operator==(const TraceKernelSel& o) const {
    return family == o.family && hist == o.hist && fast == o.fast && multi == o.multi && depth == o.depth && general == o.general;
  }
  // the selections of each family, with the fields the family does not use at their defaults
  static constexpr TraceKernelSel lockstep(bool hist, bool fast, bool multi) { return {LOCKSTEP, hist, fast, multi, 0, false}; }
  static constexpr TraceKernelSel sq(bool multi) { return {SQ, true, true, multi, 0, false}; }
  static constexpr TraceKernelSel queue(bool fast, bool multi, int depth, bool general) { return {QUEUE, true, fast, multi, depth, general}; }
  static constexpr TraceKernelSel hash(bool fast) { return {HASH, false, fast, false, 0, false}; }
  static constexpr TraceKernelSel direct(bool hist, bool fast) { return {DIRECT, hist, fast, true, 0, false}; }
  static constexpr TraceKernelSel direct_hash(bool fast) { return {DIRECT_HASH, false, fast, true, 0, false}; }
};

// launchers implemented in rthx_kernels.cu; a selection without a compiled instance fails with cudaErrorInvalidDeviceFunction
cudaError_t launch_trace_exchange(const TraceParams& p, const TraceKernelSel& k, int n_blocks, int block_threads, size_t smem_bytes,
                                  cudaStream_t stream);
cudaError_t configure_trace_kernel(size_t smem_bytes);
cudaError_t launch_fp64_peak(double* out, int n_blocks, int block_threads, int iters, cudaStream_t stream);
int trace_kernel_max_blocks_per_sm(const TraceKernelSel& k, int block_threads, size_t smem_bytes);
// Abs[k] = sum_i w[i] counts[i][k] over R rows of N, in ascending row order (rthx_trace_direct)
cudaError_t launch_direct_absorbed(const unsigned long long* counts, int R, int N, const double* w, double* absorbed, cudaStream_t stream);
// the same sum over a hashed direct tally transposed to columns: colptr [N+1], keys (source row in the low word, ascending within a
// column) and u64 counts (rthx_trace_direct_sparse)
cudaError_t launch_direct_absorbed_sparse(const long long* colptr, const unsigned long long* keys, const unsigned long long* cnt, int N, const double* w,
                                          double* absorbed, cudaStream_t stream);
constexpr size_t hash_table_bytes(int slots) { return 8 * (size_t)slots + 16; }   // keys + counts (u32 each) + occupied / fill / base words

// hashed row tally, host side of the reduction (rthx_sparse_tally.cu)
size_t tally_temp_bytes(long long n_pairs);
// sort the pairs of one row group and append (unique key, u64 total) to out_keys / out_vals at out_off; *n_unique_dev receives the count
cudaError_t tally_reduce(unsigned long long* keys, uint32_t* cnt, unsigned long long* keys_alt, uint32_t* cnt_alt, long long n_pairs, int end_bit,
                         unsigned long long* out_keys, unsigned long long* out_vals, long long* n_unique_dev, void* temp, size_t temp_bytes,
                         cudaStream_t st);
// row pointers [n_rows + 1] of the sorted unique keys (row key in the high word)
cudaError_t tally_row_ptr(const unsigned long long* keys, long long nnz, long long n_rows, long long* row_ptr, cudaStream_t st);
// rows of bin `bin` (row key y * n_bins + bin, y < n_rows): non-zeros, total and surface-gas cross tallies over the columns < n_cols.
// Row y is element row_first + y * row_stride, or rows[y] when rows != nullptr (a rows or direct trace).
cudaError_t tally_row_stats(const unsigned long long* keys, const unsigned long long* vals, const long long* row_ptr, int n_bins, int bin, int n_rows,
                            int n_cols, int n_surf, int row_first, int row_stride, const int* rows, int* nnz, unsigned long long* rowsum,
                            unsigned long long* cross, cudaStream_t st);
// the same rows as CSR at out_ptr[row]: columns < n_cols, counts, and F = count * (1 / total) (divide == false, the CSR read-out) or
// count / total (divide == true, the CSC read-out)
cudaError_t tally_row_fill(const unsigned long long* keys, const unsigned long long* vals, const long long* row_ptr, int n_bins, int bin, int n_rows,
                           int n_cols, const long long* out_ptr, const unsigned long long* rowsum, bool divide, int* cols, unsigned long long* cnt_out,
                           double* fvals, cudaStream_t st);
// merge two sorted unique (key, u64 total) sets into out_keys / out_vals (room for na + nb), summing the totals of equal keys;
// `tiles` holds 2 (tally_merge_tiles(na + nb) + 1) words, and tiles[2 * n_tiles + 1] receives the number of merged keys
long long tally_merge_tiles(long long n);
size_t tally_merge_temp_bytes(long long n_tiles);
cudaError_t tally_merge(const unsigned long long* a_keys, const unsigned long long* a_vals, long long na, const unsigned long long* b_keys,
                        const unsigned long long* b_vals, long long nb, unsigned long long* out_keys, unsigned long long* out_vals, long long* tiles,
                        void* temp, size_t temp_bytes, cudaStream_t st);
// low words of sorted transpose keys (the rows of a CSC) + base as int32 / int64; with rows != nullptr the low word y stands for
// element rows[y] (a rows or direct trace)
cudaError_t tally_key_index(const unsigned long long* keys_sorted, long long nnz, int base, const int* rows, void* out, bool i64, cudaStream_t st);

// ---- grey equilibrium solve (rthx_solve.cu) ---------------------------------------------------------------------
struct SolveMatrix {
  int kind = 0;                      // 0 dense row-major F, 1 dense col-major F (= F' row-major), 2 CSC
  const double* dense = nullptr;     // device
  size_t ld = 0;
  const long long* colptr = nullptr; // device
  const int* rowval = nullptr;
  const double* nzval = nullptr;
  long long nnz = 0;
};

struct SolveResult {
  int iterations = 0, restarts = 0, launches = 0, converged = 0, matvecs = 0;
  double residual = 0, rhs_norm = 0, total_ms = 0, matvec_ms = 0;
  long long matvec_bytes = 0;
};

size_t solve_part_doubles(int n, size_t ld);
size_t solve_vec_doubles(size_t nl, int m);
cudaError_t run_gmres(const SolveMatrix& A, int n, size_t nl, int m, int max_iters, double rtol, double atol, double* buf, double* part, double* j_host,
                      double* g_host, cudaStream_t st, cudaEvent_t e0, cudaEvent_t e1, SolveResult* out);
cudaError_t time_matvec(const SolveMatrix& A, int n, size_t nl, int m, double* buf, double* part, int reps, cudaStream_t st, cudaEvent_t e0, cudaEvent_t e1,
                        double* ms_per_pass);

}  // namespace rthx
