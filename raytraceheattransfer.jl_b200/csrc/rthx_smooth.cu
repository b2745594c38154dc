// rthx_smooth.cu — reciprocity smoothing of a dense exchange-factor matrix on the device (SURVEY.md §8(f)-2).
//
// After the trace takes ~0.2 s, the host-side alternating projection of the reference on a 10 605 x 10 605 dense matrix
// (900 MB of Float64, seconds per iteration on the CPU) dominates `mesh(N; method=:exchange)`.  This file restates the
// dense branch of src/HeatTransfer/exchangeFactorSmoothing/smoothExchangeFactors.jl on the GPU:
//   build_X    :474-490   X = (W F + (W F)')/2                         -> build_x_kernel (tile transpose, counts in)
//   hunger!    :492-499   r = X 1, u = w ./ r                           -> row sums fused into the scaling pass + u_kernel
//   scale!     :512-521   X_ij *= (u_i + u_j)/2                         -> scale_rows_kernel (one HBM pass per iteration)
//   delta_R_X  :100-118   sqrt(sum_{i<j} (X_ij (u_i-u_j))^2/(w_i^2+w_j^2)) -> delta_kernel (read-only pass, on check iterations)
//   recover_F  :546       F = X ./ r                                    -> recover_kernel
//   AP loop    :548-612   target 8 eps, floor acceptance when the contraction stalls
//   OP / DkAP  :292-318   Dykstra rounds in front of AP (the reference's default for a dense F with cross-coupling
//                         chi >= 0.4, :441-450): orthogonal projection onto {reciprocal, unit row sums} through the dual
//                         system R lambda = b (DualSolver :1-37, Jacobi-PCG, rtol 1e-14), then max(., 0) with the
//                         Dykstra correction P                         -> op_xbar / y_matvec / pcg_* / op_finalize kernels
// Every pass is HBM-bound: 16 B per matrix element per iteration (read + write of X), 8 B for a delta check.
// The sparse branch (density <= 0.25, :432-434) runs the same AP on the non-zero pattern: see "Sparse AP" at the end of this file.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <string>
#include <vector>

#include <cub/device/device_radix_sort.cuh>

#include "rthx_internal.h"

namespace rthx {

// counts (u64, row-major [N][ld]) -> row sums as doubles; one warp per row
__global__ void __launch_bounds__(256) count_rowsum_kernel(const unsigned long long* __restrict__ c, int n, size_t ld, double* __restrict__ rs) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= n) return;
  unsigned long long s = 0;
  for (int j = lane; j < n; j += 32) s += c[(size_t)row * ld + j];
  for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
  if (lane == 0) rs[row] = (double)s;
}

// X_ij = (w_i F_ij + w_j F_ji)/2 with F = counts / rowsum (rows with no tallies stay zero), 32x32 tiles through smem
// so both the (I,J) and the transposed (J,I) reads are coalesced.  F may also be given directly as doubles (rs == nullptr,
// or rs = its row sums when it still has to be row-normalised).
// XBAR: the OP form instead (Xbar_b :261-281): Xbar_ij = Y_ij (F_ij / w_i + F_ji / w_j), Y_ij = w_i^2 w_j^2 / (w_i^2 + w_j^2)
// = 1 / (a_i + a_j) with a = 1 / w^2 (reduced-mass weights, Y_mat :243-259).
template <class T, bool XBAR>
__global__ void __launch_bounds__(256) build_x_kernel(const T* __restrict__ src, size_t ld, const double* __restrict__ rs,
                                                      const double* __restrict__ w, int n, size_t ldx, double* __restrict__ X) {
  __shared__ double t[32][33];
  const int bi = blockIdx.y * 32, bj = blockIdx.x * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;   // 32 x 8
  // transposed tile: element (bj + r, bi + c) -> t[r][c]
  for (int r = ty; r < 32; r += 8) {
    const int i = bj + r, j = bi + tx;
    double v = 0.0;
    if (i < n && j < n) {
      const double d = rs ? rs[i] : 1.0;
      const double f = d > 0.0 ? (double)src[(size_t)i * ld + j] / d : 0.0;
      v = XBAR ? f / w[i] : w[i] * f;
    }
    t[r][tx] = v;
  }
  __syncthreads();
  for (int r = ty; r < 32; r += 8) {
    const int i = bi + r, j = bj + tx;
    if (i < n && j < n) {
      const double d = rs ? rs[i] : 1.0;
      const double f = d > 0.0 ? (double)src[(size_t)i * ld + j] / d : 0.0;
      if (XBAR) {
        const double wi = w[i], wj = w[j];
        const double y = 1.0 / (1.0 / (wi * wi) + 1.0 / (wj * wj));
        X[(size_t)i * ldx + j] = y * (f / wi + t[tx][r]);
      } else {
        X[(size_t)i * ldx + j] = 0.5 * (w[i] * f + t[tx][r]);
      }
    } else if (i < n && (size_t)j < ldx) {
      X[(size_t)i * ldx + j] = 0.0;                        // row padding (columns n..ldx-1) stays zero for ever
    }
  }
}

// Rows of X are padded to ldx = 16-double multiples (128-byte aligned rows; the padding holds zeros and u is padded
// with ones), so every pass streams X with aligned 16-byte accesses.  One 1024-thread block per row: 96 % of the
// measured copy bandwidth in isolation (tools/microbench/scale_pass.cu); an unpadded odd n (10 605) forces 8-byte
// accesses on misaligned rows and drops to 69 %.
constexpr int ROW_THREADS = 1024;

__device__ __forceinline__ double block_sum(double s, double* red) {
  for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  double a = 0.0;
  if (threadIdx.x == 0) for (int k = 0; k < (int)(blockDim.x >> 5); ++k) a += red[k];
  return a;
}

// plain row sums of X (first hunger!): one block per row
__global__ void __launch_bounds__(ROW_THREADS) rowsum_kernel(const double* __restrict__ X, size_t ldx, double* __restrict__ r) {
  __shared__ double red[32];
  const double2* x2 = reinterpret_cast<const double2*>(X + (size_t)blockIdx.x * ldx);
  double s = 0.0;
  for (int j = threadIdx.x; j < (int)(ldx >> 1); j += ROW_THREADS) { const double2 v = x2[j]; s += v.x + v.y; }
  const double a = block_sum(s, red);
  if (threadIdx.x == 0) r[blockIdx.x] = a;
}

// u = w ./ r on [0,n), 1 on the padding [n, ldx)
__global__ void u_kernel(const double* __restrict__ w, const double* __restrict__ r, int n, int ldx, double* __restrict__ u) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) u[i] = r[i] > 0.0 ? w[i] / r[i] : 1.0;
  else if (i < ldx) u[i] = 1.0;
}

// One AP iteration in ONE pass over HBM: X_ij *= (u_i + u_j)/2 and the new row sums r_i = sum_j X_ij.
__global__ void __launch_bounds__(ROW_THREADS) scale_rows_kernel(double* __restrict__ X, const double* __restrict__ u, size_t ldx, double* __restrict__ r) {
  __shared__ double red[32];
  const size_t row = blockIdx.x;
  const double hui = 0.5 * u[row];
  double2* x2 = reinterpret_cast<double2*>(X + row * ldx);
  const double2* u2 = reinterpret_cast<const double2*>(u);
  double s = 0.0;
  for (int j = threadIdx.x; j < (int)(ldx >> 1); j += ROW_THREADS) {
    double2 v = x2[j];
    const double2 uj = u2[j];
    v.x *= fma(0.5, uj.x, hui);
    v.y *= fma(0.5, uj.y, hui);
    x2[j] = v;
    s += v.x + v.y;
  }
  const double a = block_sum(s, red);
  if (threadIdx.x == 0) r[row] = a;
}

// delta_R^2 partial sums: sum_{j>i} (X_ij (u_i - u_j))^2 / (w_i^2 + w_j^2), one block per row -> part[row]
__global__ void __launch_bounds__(256) delta_kernel(const double* __restrict__ X, const double* __restrict__ u, const double* __restrict__ w,
                                                    int n, size_t ldx, double* __restrict__ part) {
  __shared__ double red[32];
  const size_t row = blockIdx.x;
  const double ui = u[row], wi2 = w[row] * w[row];
  double s = 0.0;
  for (int j = (int)row + 1 + threadIdx.x; j < n; j += blockDim.x) {
    const double d = X[row * ldx + j] * (ui - u[j]);
    s += d * d / (wi2 + w[j] * w[j]);
  }
  const double a = block_sum(s, red);
  if (threadIdx.x == 0) part[row] = a;
}

__global__ void __launch_bounds__(ROW_THREADS) recover_kernel(double* __restrict__ X, const double* __restrict__ r, size_t ldx) {
  const size_t row = blockIdx.x;
  const double inv = r[row] > 0.0 ? 1.0 / r[row] : 0.0;
  double2* x2 = reinterpret_cast<double2*>(X + row * ldx);
  for (int j = threadIdx.x; j < (int)(ldx >> 1); j += ROW_THREADS) { double2 v = x2[j]; v.x *= inv; v.y *= inv; x2[j] = v; }
}

// ---------------------------------------------------------------------------------------------------------------
// sparse (CSR) view of a count matrix (SURVEY.md §8(f)-3): feeds sparse(I, J, V) without moving the zeros
// ---------------------------------------------------------------------------------------------------------------
// one warp per row: number of non-zero tallies, the row total and — for cross_coupling_chi (smoothExchangeFactors.jl:212-241) —
// the tallies that couple a surface with a gas cell (exactly one of row / column index below n_surf).  The matrix may hold only
// the rows of a shard (row y = element row_first + y * row_stride) or of a rows trace (row y = element rows[y]), n_rows x n_cols with
// leading dimension ld.
__global__ void __launch_bounds__(256) row_nnz_kernel(const unsigned long long* __restrict__ c, int n_rows, int n_cols, size_t ld, int n_surf, int row_first,
                                                      int row_stride, const int* __restrict__ rows, int* __restrict__ nnz,
                                                      unsigned long long* __restrict__ rowsum, unsigned long long* __restrict__ cross) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= n_rows) return;
  int cnt = 0;
  unsigned long long s = 0, x = 0;
  const bool row_surf = (rows ? rows[row] : row_first + row * row_stride) < n_surf;
  for (int j = lane; j < n_cols; j += 32) {
    const unsigned long long v = c[(size_t)row * ld + j];
    cnt += v != 0; s += v;
    if ((j < n_surf) != row_surf) x += v;
  }
  for (int o = 16; o > 0; o >>= 1) {
    cnt += __shfl_down_sync(0xffffffffu, cnt, o); s += __shfl_down_sync(0xffffffffu, s, o); x += __shfl_down_sync(0xffffffffu, x, o);
  }
  if (lane == 0) { nnz[row] = cnt; rowsum[row] = s; if (cross) cross[row] = x; }
}

// one warp per row: write (column, count, count / rowsum) of the non-zeros in ascending column order at row_ptr[row]
__global__ void __launch_bounds__(256) row_fill_kernel(const unsigned long long* __restrict__ c, int n_rows, int n_cols, size_t ld, const long long* __restrict__ row_ptr,
                                                       const unsigned long long* __restrict__ rowsum, int* __restrict__ cols,
                                                       unsigned long long* __restrict__ vals, double* __restrict__ fvals) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= n_rows) return;
  long long base = row_ptr[row];
  const double inv = rowsum[row] ? 1.0 / (double)rowsum[row] : 0.0;
  for (int j0 = 0; j0 < n_cols; j0 += 32) {
    const int j = j0 + lane;
    const unsigned long long v = j < n_cols ? c[(size_t)row * ld + j] : 0ull;
    const unsigned m = __ballot_sync(0xffffffffu, v != 0);
    if (v != 0) {
      const long long k = base + __popc(m & ((1u << lane) - 1u));
      cols[k] = j;
      if (vals) vals[k] = v;
      if (fvals) fvals[k] = (double)v * inv;
    }
    base += __popc(m);
  }
}

cudaError_t launch_row_nnz(const unsigned long long* c, int n_rows, int n_cols, size_t ld, int n_surf, int row_first, int row_stride, const int* rows,
                           int* nnz, unsigned long long* rowsum, unsigned long long* cross, cudaStream_t st) {
  if (n_rows > 0) row_nnz_kernel<<<(n_rows + 7) / 8, 256, 0, st>>>(c, n_rows, n_cols, ld, n_surf, row_first, row_stride, rows, nnz, rowsum, cross);
  return cudaGetLastError();
}
cudaError_t launch_row_fill(const unsigned long long* c, int n_rows, int n_cols, size_t ld, const long long* row_ptr, const unsigned long long* rowsum, int* cols,
                            unsigned long long* vals, double* fvals, cudaStream_t st) {
  if (n_rows > 0) row_fill_kernel<<<(n_rows + 7) / 8, 256, 0, st>>>(c, n_rows, n_cols, ld, row_ptr, rowsum, cols, vals, fvals);
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------------------
// CSC view of a count matrix: what SparseMatrixCSC{Float64,Int} (Julia) / scipy.sparse.csc_matrix hold, emitted by the device so
// that the host neither transposes a CSR matrix nor runs sparse(I, J, V) over ~1e8 triplets (parallelRayTracing.jl:144-154 takes
// seconds there for cfg3).  Rows are cut into tiles of CSC_TILE; thread (tile, column) counts, then writes, its own run of the
// column, so both passes read the row-major matrix coalesced (consecutive threads = consecutive columns) and every column comes
// out in ascending row order.  The matrix may hold only the rows of a rows trace (n_rows x n columns, row i = element rows[i], rows
// ascending): the column view is then that of the n x n matrix whose other rows are empty.
// ---------------------------------------------------------------------------------------------------------------
constexpr int CSC_TILE = 64;

__global__ void __launch_bounds__(256) col_nnz_partial_kernel(const unsigned long long* __restrict__ c, int n_rows, int n, size_t ld, int* __restrict__ partial) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x, t = blockIdx.y;
  if (j >= n) return;
  const int i0 = t * CSC_TILE, i1 = min(n_rows, i0 + CSC_TILE);
  int cnt = 0;
  for (int i = i0; i < i1; ++i) cnt += c[(size_t)i * ld + j] != 0ull;
  partial[(size_t)t * n + j] = cnt;
}

// per column: turn the tile counts into exclusive offsets within the column, and the column total
__global__ void __launch_bounds__(256) col_offsets_kernel(int* __restrict__ partial, int n, int n_tiles, long long* __restrict__ coltotal) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  int s = 0;
  for (int t = 0; t < n_tiles; ++t) { const int v = partial[(size_t)t * n + j]; partial[(size_t)t * n + j] = s; s += v; }
  coltotal[j] = s;
}

// exclusive prefix sum of in[0..n) into out[0..n] (out[n] = total) by ONE block: every thread sums a contiguous segment, the
// 1024 segment sums are scanned in shared memory, the segment is rewritten with its running prefix.  in and out may alias.
__global__ void __launch_bounds__(1024) exclusive_scan_kernel(const long long* in, int n, long long* out) {
  __shared__ long long seg[1024];
  const int t = threadIdx.x;
  const int per = (n + 1023) / 1024;
  const int b = min(n, t * per), e = min(n, b + per);
  long long s = 0;
  for (int i = b; i < e; ++i) s += in[i];
  seg[t] = s;
  __syncthreads();
  for (int o = 1; o < 1024; o <<= 1) {
    const long long v = t >= o ? seg[t - o] : 0;
    __syncthreads();
    seg[t] += v;
    __syncthreads();
  }
  long long run = t ? seg[t - 1] : 0;
  for (int i = b; i < e; ++i) { const long long v = in[i]; out[i] = run; run += v; }
  if (t == 1023) out[n] = seg[1023];
}

template <class IDX>
__global__ void __launch_bounds__(256) col_fill_kernel(const unsigned long long* __restrict__ c, int n_rows, int n, size_t ld, const int* __restrict__ rows,
                                                       const int* __restrict__ partial, const long long* __restrict__ colptr,
                                                       const unsigned long long* __restrict__ rowsum, int index_base, IDX* __restrict__ rowval,
                                                       unsigned long long* __restrict__ vals, double* __restrict__ fvals) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x, t = blockIdx.y;
  if (j >= n) return;
  const int i0 = t * CSC_TILE, i1 = min(n_rows, i0 + CSC_TILE);
  long long k = colptr[j] + partial[(size_t)t * n + j];
  for (int i = i0; i < i1; ++i) {
    const unsigned long long v = c[(size_t)i * ld + j];
    if (v) {
      rowval[k] = (IDX)((rows ? rows[i] : i) + index_base);
      if (vals) vals[k] = v;
      if (fvals) fvals[k] = (double)v / (double)rowsum[i];      // count / row total: parallelRayTracing.jl:144-146 + row_normalize! :161-169
      ++k;
    }
  }
}

// column pointers of bin `c` (n_rows x n, leading dimension ld) into colptr[0..n] (0-based, device); partial is [n_tiles][n] ints,
// n_tiles = ceil(n_rows / 64)
cudaError_t launch_csc_count(const unsigned long long* c, int n_rows, int n, size_t ld, int* partial, long long* colptr, cudaStream_t st) {
  const int n_tiles = (n_rows + CSC_TILE - 1) / CSC_TILE;
  const dim3 grid((unsigned)((n + 255) / 256), (unsigned)n_tiles);
  col_nnz_partial_kernel<<<grid, 256, 0, st>>>(c, n_rows, n, ld, partial);
  col_offsets_kernel<<<(n + 255) / 256, 256, 0, st>>>(partial, n, n_tiles, colptr);
  exclusive_scan_kernel<<<1, 1024, 0, st>>>(colptr, n, colptr);
  return cudaGetLastError();
}
// rows (may be nullptr): element index of each of the n_rows rows
cudaError_t launch_csc_fill(const unsigned long long* c, int n_rows, int n, size_t ld, const int* rows, const int* partial, const long long* colptr,
                            const unsigned long long* rowsum, int index_base, void* rowval, bool rowval_i64, unsigned long long* vals, double* fvals,
                            cudaStream_t st) {
  const int n_tiles = (n_rows + CSC_TILE - 1) / CSC_TILE;
  const dim3 grid((unsigned)((n + 255) / 256), (unsigned)n_tiles);
  if (rowval_i64) col_fill_kernel<long long><<<grid, 256, 0, st>>>(c, n_rows, n, ld, rows, partial, colptr, rowsum, index_base, (long long*)rowval, vals, fvals);
  else col_fill_kernel<int><<<grid, 256, 0, st>>>(c, n_rows, n, ld, rows, partial, colptr, rowsum, index_base, (int*)rowval, vals, fvals);
  return cudaGetLastError();
}
// colptr += base (1-based pointers for Julia), in place
__global__ void add_base_kernel(long long* p, int n, long long base) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] += base;
}
cudaError_t launch_add_base(long long* p, int n, long long base, cudaStream_t st) {
  add_base_kernel<<<(n + 255) / 256, 256, 0, st>>>(p, n, base);
  return cudaGetLastError();
}

struct SmoothResult { int iters; double delta, delta_init; double ms_total, ms_per_iter; int launches; int converged; };

// non-zeros of the leading n x n block of a matrix (u64 counts or doubles): the density enters AP's floor-aware acceptance
template <class T>
__global__ void __launch_bounds__(256) nnz_count_kernel(const T* __restrict__ src, int n, size_t ld, unsigned long long* __restrict__ out) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= n) return;
  unsigned int cnt = 0;
  for (int j = lane; j < n; j += 32) cnt += src[(size_t)row * ld + j] != (T)0;
  for (int o = 16; o > 0; o >>= 1) cnt += __shfl_down_sync(0xffffffffu, cnt, o);
  if (lane == 0 && cnt) atomicAdd(out, (unsigned long long)cnt);
}

// The AP iteration with the reference's stopping rule (smoothExchangeFactors.jl:548-612), shared by the dense and the sparse
// form: `step()` enqueues one iteration (scaling pass + u = w ./ r), `delta_now(&d)` returns delta_R_X of the current iterate.
// `guard` is the floor below which a stalled contraction is accepted.  Returns the iterations run and the final delta.
struct ApLoop { int iters; double delta, delta_init; bool floor_accepted; };
template <class Step, class Delta>
static cudaError_t ap_loop(int max_iters, double target, double guard, Step step, Delta delta_now, ApLoop* out) {
  cudaError_t e;
  double delta = 0;
  if ((e = delta_now(&delta)) != cudaSuccess) return e;
  const double delta_init = delta;
  double best = delta, delta_prev = delta, rho_est = 0.5;
  int k = 0, k_next = 1, flat = 0, checks = 0, k_prev = 0;
  bool floor_accepted = false;
  while (k < max_iters && delta > target) {
    if ((e = step()) != cudaSuccess) return e;
    ++k;
    if (k >= k_next || k == max_iters) {
      if ((e = delta_now(&delta)) != cudaSuccess) return e;
      // the reference's stopping rule (smoothExchangeFactors.jl:578-590): contraction estimate and the flat count start with
      // the third check; a stalled contraction is accepted only below the guard, otherwise the loop runs to max_iters
      ++checks;
      if (checks >= 3) {
        rho_est = std::min(std::max(std::pow(delta / delta_prev, 1.0 / std::max(k - k_prev, 1)), 0.5), 0.9999);
        flat = delta >= best * (1 - 1e-3) ? flat + 1 : 0;
      }
      best = std::min(best, delta);
      if (delta < guard && (rho_est > 0.99 || flat >= 3)) { floor_accepted = true; break; }
      k_prev = k; delta_prev = delta;
      k_next = k + std::min(32, std::max(1, k));             // 1,2,4,...,32 then every 32 iterations
    }
  }
  out->iters = k; out->delta = delta; out->delta_init = delta_init; out->floor_accepted = floor_accepted;
  return cudaSuccess;
}

// Runs AP on the device.  `src_counts` (u64, leading dimension ld) or `src_F` (doubles; `src_rs` = its row sums when it
// still has to be row-normalised, else nullptr) is a DEVICE pointer; X (n*ldx doubles) and the work vectors are device
// scratch owned by the caller.  On return X holds F_smooth.
cudaError_t run_ap(const unsigned long long* src_counts, const double* src_F, const double* src_rs, size_t ld, const double* w_dev, int n, size_t ldx, int max_iters, double target,
                   double* X, double* rs, double* r, double* u, double* part, std::vector<double>& part_host, cudaStream_t st, cudaEvent_t e0,
                   cudaEvent_t e1, SmoothResult* out) {
  cudaError_t e;
  int launches = 0;
  const dim3 tg((unsigned)((ldx + 31) / 32), (n + 31) / 32);   // x covers the row padding too
  if ((e = cudaEventRecord(e0, st)) != cudaSuccess) return e;
  if (src_counts) {
    count_rowsum_kernel<<<(n + 7) / 8, 256, 0, st>>>(src_counts, n, ld, rs);
    build_x_kernel<unsigned long long, false><<<tg, 256, 0, st>>>(src_counts, ld, rs, w_dev, n, ldx, X);
    launches += 2;
  } else {
    build_x_kernel<double, false><<<tg, 256, 0, st>>>(src_F, ld, src_rs, w_dev, n, ldx, X);
    launches += 1;
  }
  rowsum_kernel<<<n, ROW_THREADS, 0, st>>>(X, ldx, r);
  u_kernel<<<(unsigned)((ldx + 255) / 256), 256, 0, st>>>(w_dev, r, n, (int)ldx, u);
  launches += 2;
  auto delta_now = [&](double* d) -> cudaError_t {
    delta_kernel<<<n, 256, 0, st>>>(X, u, w_dev, n, ldx, part);
    ++launches;
    cudaError_t ee = cudaMemcpyAsync(part_host.data(), part, sizeof(double) * n, cudaMemcpyDeviceToHost, st);
    if (ee != cudaSuccess) return ee;
    if ((ee = cudaStreamSynchronize(st)) != cudaSuccess) return ee;
    double s = 0;
    for (int i = 0; i < n; ++i) s += part_host[i];
    *d = std::sqrt(s);
    return cudaSuccess;
  };
  // floor-aware acceptance (smoothExchangeFactors.jl:558-560): guard = sqrt(N / nz_over_N) * target = target / sqrt(density)
  double guard = target;
  {
    unsigned long long* nz_dev = reinterpret_cast<unsigned long long*>(part);   // part is free until the first delta check
    if ((e = cudaMemsetAsync(nz_dev, 0, sizeof(unsigned long long), st)) != cudaSuccess) return e;
    if (src_counts) nnz_count_kernel<unsigned long long><<<(n + 7) / 8, 256, 0, st>>>(src_counts, n, ld, nz_dev);
    else nnz_count_kernel<double><<<(n + 7) / 8, 256, 0, st>>>(src_F, n, ld, nz_dev);
    ++launches;
    unsigned long long nz = 0;
    if ((e = cudaMemcpyAsync(&nz, nz_dev, sizeof(nz), cudaMemcpyDeviceToHost, st)) != cudaSuccess) return e;
    if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return e;
    if (nz > 0) guard = target * std::sqrt((double)n * (double)n / (double)nz);
  }
  auto step = [&]() -> cudaError_t {
    scale_rows_kernel<<<n, ROW_THREADS, 0, st>>>(X, u, ldx, r);
    u_kernel<<<(unsigned)((ldx + 255) / 256), 256, 0, st>>>(w_dev, r, n, (int)ldx, u);
    launches += 2;
    return cudaSuccess;
  };
  ApLoop lp{};
  if ((e = ap_loop(max_iters, target, guard, step, delta_now, &lp)) != cudaSuccess) return e;
  recover_kernel<<<n, ROW_THREADS, 0, st>>>(X, r, ldx);
  ++launches;
  if ((e = cudaEventRecord(e1, st)) != cudaSuccess) return e;
  if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return e;
  float ms = 0;
  cudaEventElapsedTime(&ms, e0, e1);
  const int k = lp.iters;
  out->iters = k; out->delta = lp.delta; out->delta_init = lp.delta_init; out->ms_total = ms;
  out->ms_per_iter = k > 0 ? ms / k : 0.0; out->launches = launches;
  out->converged = (lp.delta <= target || lp.floor_accepted) ? 1 : 0;     // else the reference warns "AP reached max_iters" (:605-607)
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------------------
// Dykstra rounds (OP) in front of AP — smoothExchangeFactors.jl:1-37 (DualSolver, solve_R), :261-318 (Xbar_b, OP, DkAP)
// ---------------------------------------------------------------------------------------------------------------
// a = 1 / w^2 on [0,n)
__global__ void inv_sq_kernel(const double* __restrict__ w, int n, double* __restrict__ a) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) a[i] = 1.0 / (w[i] * w[i]);
}

// out_i = sum_j Y_ij v_j (+ rowsumY_i v_i when rowsumY != nullptr: R = Y + Diagonal(Y 1), Rmul! :13), Y_ij = 1/(a_i + a_j)
// formed on the fly — no N^2 matrix is stored or streamed.  v == nullptr means v = 1 (the row sums of Y).
__global__ void __launch_bounds__(256) y_matvec_kernel(const double* __restrict__ a, const double* __restrict__ v, const double* __restrict__ rowsumY,
                                                       int n, double* __restrict__ out) {
  __shared__ double red[32];
  const int i = blockIdx.x;
  const double ai = a[i];
  double s = 0.0;
  for (int j = threadIdx.x; j < n; j += blockDim.x) s += (v ? v[j] : 1.0) / (ai + a[j]);
  const double t = block_sum(s, red);
  if (threadIdx.x == 0) out[i] = rowsumY ? fma(rowsumY[i], v[i], t) : t;
}

// 1024-thread single-block reductions for the PCG scalars (fixed order: bit-reproducible)
__device__ __forceinline__ double block_allsum_1024(double s, double* red) {
  for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
  __syncthreads();                                     // red may still be read from the previous reduction
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  double a = 0.0;
  for (int k = 0; k < 32; ++k) a += red[k];
  return a;
}

// dinv = 1 / (Y_ii + rowsumY_i), Y_ii = w_i^2 / 2 = 1 / (2 a_i)   (DualSolver :7-11)
__global__ void dinv_kernel(const double* __restrict__ a, const double* __restrict__ rowsumY, int n, double* __restrict__ dinv) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dinv[i] = 1.0 / (0.5 / a[i] + rowsumY[i]);
}

// b = rowsum - w (OP right-hand side, Xbar_b) or b = w .* (rowsum - 1) (delta_perp :DYK, :139)
__global__ void op_rhs_kernel(const double* __restrict__ rowsum, const double* __restrict__ w, int n, int dyk, double* __restrict__ b) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) b[i] = dyk ? w[i] * (rowsum[i] - 1.0) : rowsum[i] - w[i];
}

// solve_R :15-37 — x = 0, r = b, z = dinv r, p = z; sc[0] = r.z, sc[1] = |r|^2, sc[3] = |b|^2
__global__ void __launch_bounds__(1024) pcg_init_kernel(int n, const double* __restrict__ b, const double* __restrict__ dinv, double* __restrict__ x,
                                                        double* __restrict__ r, double* __restrict__ z, double* __restrict__ p, double* __restrict__ sc) {
  __shared__ double red[32];
  double rz = 0.0, bb = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const double bi = b[i], zi = dinv[i] * bi;
    x[i] = 0.0; r[i] = bi; z[i] = zi; p[i] = zi;
    rz = fma(bi, zi, rz); bb = fma(bi, bi, bb);
  }
  rz = block_allsum_1024(rz, red);
  bb = block_allsum_1024(bb, red);
  if (threadIdx.x == 0) { sc[0] = rz; sc[1] = bb; sc[3] = bb; }
}

// one PCG iteration after Ap = R p: alpha = rz / p.Ap; x += alpha p; r -= alpha Ap; z = dinv r; beta = r.z / rz; p = z + beta p
__global__ void __launch_bounds__(1024) pcg_step_kernel(int n, const double* __restrict__ dinv, const double* __restrict__ Ap, double* __restrict__ x,
                                                        double* __restrict__ r, double* __restrict__ z, double* __restrict__ p, double* __restrict__ sc) {
  __shared__ double red[32];
  double pap = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) pap = fma(p[i], Ap[i], pap);
  pap = block_allsum_1024(pap, red);
  const double rz = sc[0];
  const double alpha = rz / pap;
  double rn = 0.0, rzn = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    x[i] = fma(alpha, p[i], x[i]);
    const double ri = fma(-alpha, Ap[i], r[i]);
    const double zi = dinv[i] * ri;
    r[i] = ri; z[i] = zi;
    rn = fma(ri, ri, rn); rzn = fma(ri, zi, rzn);
  }
  rn = block_allsum_1024(rn, red);
  rzn = block_allsum_1024(rzn, red);
  const double beta = rzn / rz;
  for (int i = threadIdx.x; i < n; i += blockDim.x) p[i] = fma(beta, p[i], z[i]);
  __syncthreads();
  if (threadIdx.x == 0) { sc[0] = rzn; sc[1] = rn; }
}

// sc[2] = u . v (single block)
__global__ void __launch_bounds__(1024) dot_kernel(int n, const double* __restrict__ u, const double* __restrict__ v, double* __restrict__ sc) {
  __shared__ double red[32];
  double s = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) s = fma(u[i], v[i], s);
  s = block_allsum_1024(s, red);
  if (threadIdx.x == 0) sc[2] = s;
}

// OP :292-297 + the Dykstra update of DkAP :306-313, in place on the Xbar buffer, one block per row:
//   G = (Xbar - Y .* (lambda_i + lambda_j)) / w_i;  F = max(G + P, 0);  P = G + P - F;  rs_i = sum_j F_ij
__global__ void __launch_bounds__(ROW_THREADS) op_finalize_kernel(double* __restrict__ Xb, double* __restrict__ P, const double* __restrict__ w,
                                                                  const double* __restrict__ a, const double* __restrict__ lam, int n, size_t ldx,
                                                                  double* __restrict__ rs) {
  __shared__ double red[32];
  const size_t row = blockIdx.x;
  const double ai = a[row], li = lam[row], inv_wi = 1.0 / w[row];
  double s = 0.0;
  for (int j = threadIdx.x; j < n; j += ROW_THREADS) {
    const double y = 1.0 / (ai + a[j]);
    const double g = (Xb[row * ldx + j] - y * (li + lam[j])) * inv_wi;
    const double t = P ? g + P[row * ldx + j] : g;
    const double f = fmax(t, 0.0);
    if (P) P[row * ldx + j] = t - f;
    Xb[row * ldx + j] = f;
    s += f;
  }
  const double tot = block_sum(s, red);
  if (threadIdx.x == 0) rs[row] = tot;
}

struct DykstraResult { int rounds; int pcg_iters; double delta; double ms; int launches; };

// Jacobi-PCG on R lambda = b (solve_R :15-37: rtol 1e-14, maxiter 200).  vec: a, rowsumY, dinv, b, x, r, z, p, Ap
static cudaError_t pcg_solve(int n, const double* a, const double* rowsumY, const double* dinv, const double* b, double* x, double* r, double* z,
                             double* p, double* Ap, double* sc, cudaStream_t st, int* iters, int* launches) {
  cudaError_t e;
  pcg_init_kernel<<<1, 1024, 0, st>>>(n, b, dinv, x, r, z, p, sc);
  ++*launches;
  double h[4];
  if ((e = cudaMemcpyAsync(h, sc, sizeof(h), cudaMemcpyDeviceToHost, st)) != cudaSuccess) return e;
  if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return e;
  const double bn = std::sqrt(h[3]);
  *iters = 0;
  if (bn == 0.0) return cudaSuccess;
  for (int it = 1; it <= 200; ++it) {
    y_matvec_kernel<<<n, 256, 0, st>>>(a, p, rowsumY, n, Ap);
    pcg_step_kernel<<<1, 1024, 0, st>>>(n, dinv, Ap, x, r, z, p, sc);
    *launches += 2;
    *iters = it;
    if ((e = cudaMemcpyAsync(h, sc, sizeof(double) * 2, cudaMemcpyDeviceToHost, st)) != cudaSuccess) return e;
    if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return e;
    if (std::sqrt(h[1]) <= 1e-14 * bn) break;
  }
  return cudaGetLastError();
}

// k_dykstra rounds of OP + clipping.  Source as in run_ap.  B (and C, P when k_dykstra > 1) are n*ldx device buffers;
// vec holds 10 vectors of ldx doubles + 8 scalars.  On return *F_out (B or C) holds the clipped iterate and rs_out its row
// sums; the caller hands both to run_ap, which renormalises the rows (DkAP :316) and polishes with AP (:317).
cudaError_t run_dykstra(const unsigned long long* src_counts, const double* src_F, size_t ld, const double* w_dev, int n, size_t ldx, int k_dykstra,
                        double* B, double* C, double* P, double* vec, cudaStream_t st, cudaEvent_t e0, cudaEvent_t e1, double** F_out, double** rs_out,
                        DykstraResult* out) {
  cudaError_t e;
  double *a = vec, *rowsumY = a + ldx, *dinv = rowsumY + ldx, *b = dinv + ldx, *lam = b + ldx, *r = lam + ldx, *z = r + ldx, *p = z + ldx,
         *Ap = p + ldx, *rs = Ap + ldx, *sc = rs + ldx;
  int launches = 0, pcg_total = 0;
  const int vb = (n + 255) / 256;
  const dim3 tg((unsigned)((ldx + 31) / 32), (n + 31) / 32);
  if ((e = cudaEventRecord(e0, st)) != cudaSuccess) return e;
  inv_sq_kernel<<<vb, 256, 0, st>>>(w_dev, n, a);
  y_matvec_kernel<<<n, 256, 0, st>>>(a, nullptr, nullptr, n, rowsumY);
  dinv_kernel<<<vb, 256, 0, st>>>(a, rowsumY, n, dinv);
  launches += 3;
  if (P && (e = cudaMemsetAsync(P, 0, sizeof(double) * (size_t)n * ldx, st)) != cudaSuccess) return e;
  double delta = INFINITY;
  double* cur = nullptr;
  int k = 1;
  for (; k <= k_dykstra; ++k) {
    double* dst = (k & 1) ? B : C;
    if (k == 1 && src_counts) {
      count_rowsum_kernel<<<(n + 7) / 8, 256, 0, st>>>(src_counts, n, ld, rs);
      build_x_kernel<unsigned long long, true><<<tg, 256, 0, st>>>(src_counts, ld, rs, w_dev, n, ldx, dst);
      launches += 2;
    } else if (k == 1) {
      build_x_kernel<double, true><<<tg, 256, 0, st>>>(src_F, ld, nullptr, w_dev, n, ldx, dst);
      ++launches;
    } else {
      build_x_kernel<double, true><<<tg, 256, 0, st>>>(cur, ldx, nullptr, w_dev, n, ldx, dst);
      ++launches;
    }
    rowsum_kernel<<<n, ROW_THREADS, 0, st>>>(dst, ldx, rs);
    op_rhs_kernel<<<vb, 256, 0, st>>>(rs, w_dev, n, 0, b);
    launches += 2;
    int it = 0;
    if ((e = pcg_solve(n, a, rowsumY, dinv, b, lam, r, z, p, Ap, sc, st, &it, &launches)) != cudaSuccess) return e;
    pcg_total += it;
    op_finalize_kernel<<<n, ROW_THREADS, 0, st>>>(dst, k_dykstra > 1 ? P : nullptr, w_dev, a, lam, n, ldx, rs);
    ++launches;
    cur = dst;
    if (k % 5 == 0 || k == k_dykstra) {                        // delta_perp(:DYK) :136-142
      op_rhs_kernel<<<vb, 256, 0, st>>>(rs, w_dev, n, 1, b);
      ++launches;
      if ((e = pcg_solve(n, a, rowsumY, dinv, b, lam, r, z, p, Ap, sc, st, &it, &launches)) != cudaSuccess) return e;
      dot_kernel<<<1, 1024, 0, st>>>(n, b, lam, sc);
      ++launches;
      double d2 = 0;
      if ((e = cudaMemcpyAsync(&d2, sc + 2, sizeof(double), cudaMemcpyDeviceToHost, st)) != cudaSuccess) return e;
      if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return e;
      delta = std::sqrt(std::max(d2, 0.0));
    }
    if (delta < 8 * 2.220446049250313e-16) { ++k; break; }
  }
  if ((e = cudaEventRecord(e1, st)) != cudaSuccess) return e;
  if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return e;
  float ms = 0;
  cudaEventElapsedTime(&ms, e0, e1);
  *F_out = cur; *rs_out = rs;
  out->rounds = k - 1; out->pcg_iters = pcg_total; out->delta = delta; out->ms = ms; out->launches = launches;
  return cudaGetLastError();
}

// timing helper for the roofline: `reps` back-to-back scaling passes with u = 1 (X unchanged), returns ms per pass
cudaError_t time_scale_pass(double* X, double* u, double* r, int n, size_t ldx, int reps, cudaStream_t st, cudaEvent_t e0, cudaEvent_t e1, double* ms_per_pass) {
  cudaError_t e;
  scale_rows_kernel<<<n, ROW_THREADS, 0, st>>>(X, u, ldx, r);
  if ((e = cudaEventRecord(e0, st)) != cudaSuccess) return e;
  for (int i = 0; i < reps; ++i) scale_rows_kernel<<<n, ROW_THREADS, 0, st>>>(X, u, ldx, r);
  if ((e = cudaEventRecord(e1, st)) != cudaSuccess) return e;
  if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return e;
  float ms = 0;
  cudaEventElapsedTime(&ms, e0, e1);
  *ms_per_pass = ms / reps;
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------------------
// Sparse AP: the branch of smooth_F for density <= 0.25 (smoothExchangeFactors.jl:432-434, AP :548-612 on the non-zero
// pattern).  F arrives as CSC (uploaded, or compacted from the resident counts by csc_count / csc_fill); its transpose (the
// CSR of F) comes from a radix sort of (row, column) keys, so the order within a row is fixed.  X = (W F + (W F)')/2 lives on
// the union pattern of F and F' as CSR with ascending columns and is exactly symmetric, so F_smooth = X ./ r leaves as CSC
// without a transpose: colptr = X's row pointers, rowval = X's columns, nzval[p] = X[p] / r[col[p]].
// One iteration is one pass over X: 8 B value read + 8 B write + 4 B column index per entry, plus the row pointers; u
// (8 n bytes) is gathered from L2.
// ---------------------------------------------------------------------------------------------------------------

// CSC of F -> transpose keys (row << 32 | column) and the non-zeros per row of F (atomic counts: the totals are deterministic)
__global__ void __launch_bounds__(256) csc_keys_kernel(const long long* __restrict__ colptr, const int* __restrict__ rowval, int n,
                                                       unsigned long long* __restrict__ keys, unsigned long long* __restrict__ row_cnt) {
  const int j = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (j >= n) return;
  for (long long p = colptr[j] + lane; p < colptr[j + 1]; p += 32) {
    const int i = rowval[p];
    keys[p] = ((unsigned long long)i << 32) | (unsigned)j;
    atomicAdd(row_cnt + i, 1ull);
  }
}

// Row i of X is the union of row i of F (sorted keys [rptr[i], rptr[i+1]), column in the low word) and column i of F (rowval
// [colptr[i], colptr[i+1]), ascending); one thread per row merges the two lists.  FILL == false counts the union into xptr[i];
// FILL == true writes X_ij = (w_i F_ij + w_j F_ji) / 2.  X_ji is the same expression with the two products swapped; the
// products are rounded on their own (no FMA contraction) so that the sum, and with it X, is exactly symmetric.
template <bool FILL>
__global__ void __launch_bounds__(256) x_merge_kernel(int n, const long long* __restrict__ colptr, const int* __restrict__ rowval,
                                                      const double* __restrict__ val, const long long* __restrict__ rptr,
                                                      const unsigned long long* __restrict__ keys, const double* __restrict__ kval,
                                                      const double* __restrict__ w, long long* __restrict__ xptr, int* __restrict__ xcol,
                                                      double* __restrict__ xval) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  long long a = rptr[i], b = colptr[i], k = FILL ? xptr[i] : 0;
  const long long ae = rptr[i + 1], be = colptr[i + 1];
  const double wi = FILL ? w[i] : 0.0;
  while (a < ae || b < be) {
    const int ja = a < ae ? (int)(keys[a] & 0xffffffffull) : 0x7fffffff;
    const int jb = b < be ? rowval[b] : 0x7fffffff;
    const int j = min(ja, jb);
    if (FILL) {
      const double fij = ja == j ? kval[a] : 0.0, fji = jb == j ? val[b] : 0.0;
      xcol[k] = j;
      xval[k] = 0.5 * __dadd_rn(__dmul_rn(wi, fij), __dmul_rn(w[j], fji));
    }
    ++k;
    a += ja == j;
    b += jb == j;
  }
  if (!FILL) xptr[i] = k;
}

// One warp per row of X: (SCALE) X_p *= (u_i + u_col(p))/2, then r_i = sum of the row — lane-strided partial sums and a fixed
// shuffle tree, so the order is the same on every call — and u'_i = w_i / r_i (1 for an empty row) into the OTHER u buffer:
// the rows still being scaled keep reading the old u.  SCALE == false: the first hunger! (row sums of X as built).
template <bool SCALE>
__global__ void __launch_bounds__(256) csr_scale_kernel(int n, const long long* __restrict__ xptr, const int* __restrict__ xcol,
                                                        double* __restrict__ xval, const double* __restrict__ u, const double* __restrict__ w,
                                                        double* __restrict__ r, double* __restrict__ u_next) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= n) return;
  const long long e = xptr[row + 1];
  const double hui = SCALE ? 0.5 * u[row] : 0.0;
  double s = 0.0;
  for (long long p = xptr[row] + lane; p < e; p += 32) {
    double v = xval[p];
    if (SCALE) {
      v *= fma(0.5, u[xcol[p]], hui);       // = (u_i + u_j)/2 rounded once: the same factor for X_ij and X_ji
      xval[p] = v;
    }
    s += v;
  }
  for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
  if (lane == 0) { r[row] = s; u_next[row] = s > 0.0 ? w[row] / s : 1.0; }
}

// delta_R_X^2 per row over the stored upper-triangle entries: sum_{j>i} (X_ij (u_i - u_j))^2 / (w_i^2 + w_j^2) -> part[row]
__global__ void __launch_bounds__(256) csr_delta_kernel(int n, const long long* __restrict__ xptr, const int* __restrict__ xcol,
                                                        const double* __restrict__ xval, const double* __restrict__ u, const double* __restrict__ w,
                                                        double* __restrict__ part) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= n) return;
  const double ui = u[row], wi2 = w[row] * w[row];
  const long long e = xptr[row + 1];
  double s = 0.0;
  for (long long p = xptr[row] + lane; p < e; p += 32) {
    const int j = xcol[p];
    if (j > row) {
      const double d = xval[p] * (ui - u[j]);
      s += d * d / (wi2 + w[j] * w[j]);
    }
  }
  for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
  if (lane == 0) part[row] = s;
}

// *out = sum of part[0..n) in a fixed order (one block): the delta check moves 8 bytes to the host, not n partial sums
__global__ void __launch_bounds__(1024) sum_kernel(const double* __restrict__ part, int n, double* __restrict__ out) {
  __shared__ double red[32];
  double s = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) s += part[i];
  s = block_allsum_1024(s, red);
  if (threadIdx.x == 0) *out = s;
}

// recover_F (:537-546) written straight as the CSC of F_smooth: nzval[p] = X[p] / r[col[p]], in place
__global__ void __launch_bounds__(256) csr_recover_kernel(long long nnz, const int* __restrict__ xcol, const double* __restrict__ r, double* __restrict__ xval) {
  for (long long p = blockIdx.x * (long long)blockDim.x + threadIdx.x; p < nnz; p += (long long)gridDim.x * blockDim.x) {
    const double d = r[xcol[p]];
    xval[p] = d > 0.0 ? xval[p] / d : 0.0;
  }
}

template <class IDX>
__global__ void __launch_bounds__(256) index_out_kernel(const int* __restrict__ col, long long nnz, int base, IDX* __restrict__ out) {
  for (long long p = blockIdx.x * (long long)blockDim.x + threadIdx.x; p < nnz; p += (long long)gridDim.x * blockDim.x) out[p] = (IDX)col[p] + base;
}

static unsigned flat_blocks(long long nnz) { return (unsigned)std::max<long long>(1, std::min<long long>((nnz + 255) / 256, 148 * 32)); }
static int sort_end_bit(int n) { int b = 1; while ((1ll << b) < (long long)n) ++b; return 32 + b; }

size_t sparse_sort_temp_bytes(int nnz, int n) {
  size_t bytes = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, bytes, (const unsigned long long*)nullptr, (unsigned long long*)nullptr, (const double*)nullptr,
                                  (double*)nullptr, nnz, 0, sort_end_bit(n));
  return bytes;
}

// CSR of F from its CSC: rptr [n+1] (row pointers), keys_sorted / val_sorted [nnz] (row-major order, ascending columns)
cudaError_t sparse_transpose(int n, int nnz, const long long* colptr, const int* rowval, const double* val, unsigned long long* keys,
                             unsigned long long* keys_sorted, double* val_sorted, long long* rptr, void* temp, size_t temp_bytes, cudaStream_t st) {
  cudaError_t e;
  if ((e = cudaMemsetAsync(rptr, 0, sizeof(long long) * ((size_t)n + 1), st)) != cudaSuccess) return e;
  csc_keys_kernel<<<(n + 7) / 8, 256, 0, st>>>(colptr, rowval, n, keys, reinterpret_cast<unsigned long long*>(rptr));
  exclusive_scan_kernel<<<1, 1024, 0, st>>>(rptr, n, rptr);
  if (nnz > 0 && (e = cub::DeviceRadixSort::SortPairs(temp, temp_bytes, keys, keys_sorted, val, val_sorted, nnz, 0, sort_end_bit(n), st)) != cudaSuccess)
    return e;
  return cudaGetLastError();
}

// row pointers of X (union pattern) into xptr [n+1]
cudaError_t launch_x_count(int n, const long long* colptr, const int* rowval, const long long* rptr, const unsigned long long* keys_sorted, long long* xptr,
                           cudaStream_t st) {
  x_merge_kernel<false><<<(n + 255) / 256, 256, 0, st>>>(n, colptr, rowval, nullptr, rptr, keys_sorted, nullptr, nullptr, xptr, nullptr, nullptr);
  exclusive_scan_kernel<<<1, 1024, 0, st>>>(xptr, n, xptr);
  return cudaGetLastError();
}

cudaError_t launch_x_fill(int n, const long long* colptr, const int* rowval, const double* val, const long long* rptr, const unsigned long long* keys_sorted,
                          const double* val_sorted, const double* w, long long* xptr, int* xcol, double* xval, cudaStream_t st) {
  x_merge_kernel<true><<<(n + 255) / 256, 256, 0, st>>>(n, colptr, rowval, val, rptr, keys_sorted, val_sorted, w, xptr, xcol, xval);
  return cudaGetLastError();
}

// AP on the CSR iterate X (n rows, nnz_x entries); nnz_f = non-zeros of F for the floor guard.  vec: r, u0, u1, part [n each]
// + 8 scalars.  On return xval holds the values of F_smooth as CSC (see above).  Timing is the caller's.
cudaError_t run_ap_sparse(int n, long long nnz_f, long long nnz_x, const long long* xptr, const int* xcol, double* xval, const double* w, double* vec,
                          int max_iters, double target, cudaStream_t st, SmoothResult* out) {
  cudaError_t e;
  double *r = vec, *u = r + n, *un = u + n, *part = un + n, *sc = part + n;
  const unsigned rb = (unsigned)((n + 7) / 8);
  int launches = 1;
  csr_scale_kernel<false><<<rb, 256, 0, st>>>(n, xptr, xcol, xval, nullptr, w, r, u);     // r = X 1, u = w ./ r
  auto delta_now = [&](double* d) -> cudaError_t {
    csr_delta_kernel<<<rb, 256, 0, st>>>(n, xptr, xcol, xval, u, w, part);
    sum_kernel<<<1, 1024, 0, st>>>(part, n, sc);
    launches += 2;
    double s = 0;
    cudaError_t ee = cudaMemcpyAsync(&s, sc, sizeof(double), cudaMemcpyDeviceToHost, st);
    if (ee != cudaSuccess) return ee;
    if ((ee = cudaStreamSynchronize(st)) != cudaSuccess) return ee;
    *d = std::sqrt(s);
    return cudaSuccess;
  };
  auto step = [&]() -> cudaError_t {
    csr_scale_kernel<true><<<rb, 256, 0, st>>>(n, xptr, xcol, xval, u, w, r, un);
    std::swap(u, un);
    ++launches;
    return cudaSuccess;
  };
  // floor-aware acceptance (smoothExchangeFactors.jl:558-560): guard = target * sqrt(n^2 / nnz_F)
  const double guard = nnz_f > 0 ? target * std::sqrt((double)n * (double)n / (double)nnz_f) : target;
  ApLoop lp{};
  if ((e = ap_loop(max_iters, target, guard, step, delta_now, &lp)) != cudaSuccess) return e;
  if (nnz_x > 0) { csr_recover_kernel<<<flat_blocks(nnz_x), 256, 0, st>>>(nnz_x, xcol, r, xval); ++launches; }
  out->iters = lp.iters; out->delta = lp.delta; out->delta_init = lp.delta_init; out->launches = launches;
  out->converged = (lp.delta <= target || lp.floor_accepted) ? 1 : 0;
  out->ms_total = out->ms_per_iter = 0.0;
  return cudaGetLastError();
}

// timing helper: `reps` back-to-back sparse scaling passes with u = 1 (the factor is exactly 1: X is unchanged)
cudaError_t time_sparse_pass(int n, const long long* xptr, const int* xcol, double* xval, const double* w, double* vec, int reps, cudaStream_t st,
                             cudaEvent_t e0, cudaEvent_t e1, double* ms_per_pass) {
  cudaError_t e;
  double *r = vec, *u = r + n, *un = u + n;
  std::vector<double> ones((size_t)n, 1.0);
  if ((e = cudaMemcpyAsync(u, ones.data(), sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, st)) != cudaSuccess) return e;
  const unsigned rb = (unsigned)((n + 7) / 8);
  csr_scale_kernel<true><<<rb, 256, 0, st>>>(n, xptr, xcol, xval, u, w, r, un);
  if ((e = cudaEventRecord(e0, st)) != cudaSuccess) return e;
  for (int i = 0; i < reps; ++i) csr_scale_kernel<true><<<rb, 256, 0, st>>>(n, xptr, xcol, xval, u, w, r, un);
  if ((e = cudaEventRecord(e1, st)) != cudaSuccess) return e;
  if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return e;
  float ms = 0;
  cudaEventElapsedTime(&ms, e0, e1);
  *ms_per_pass = ms / reps;
  return cudaGetLastError();
}

// column indices of the resident F_smooth for the caller: + index_base, as int32 or int64
cudaError_t launch_index_out(const int* col, long long nnz, int base, void* out, bool i64, cudaStream_t st) {
  if (nnz <= 0) return cudaSuccess;
  if (i64) index_out_kernel<long long><<<flat_blocks(nnz), 256, 0, st>>>(col, nnz, base, (long long*)out);
  else index_out_kernel<int><<<flat_blocks(nnz), 256, 0, st>>>(col, nnz, base, (int*)out);
  return cudaGetLastError();
}

}  // namespace rthx
