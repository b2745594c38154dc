// rthx_sparse_tally.cu — device side of the hashed row tally after the trace (rthx_trace_exchange_sparse): the (row key << 32 |
// column, count) pairs the HASH trace kernels flushed are radix-sorted and reduced by key into u64 totals, so the only
// nondeterminism of the tally (the order in which blocks reserved buffer space) is gone; row pointers come from the sorted keys,
// and the read-outs of the resident counts (CSR / CSC / row statistics / the sparse smoothing's F) are formed from them with the
// value formulas of the dense read-outs (rthx_smooth.cu), so that they agree bit for bit.
#include <cub/device/device_radix_sort.cuh>
#include <cub/block/block_scan.cuh>
#include <cub/device/device_reduce.cuh>
#include <cub/device/device_scan.cuh>
#include <cuda/std/functional>
#include <thrust/iterator/transform_iterator.h>

#include "rthx_internal.h"

namespace rthx {

namespace {
struct WidenU32 {
  __host__ __device__ unsigned long long operator()(uint32_t v) const { return v; }
};

__global__ void __launch_bounds__(256) row_ptr_kernel(const unsigned long long* __restrict__ keys, long long nnz, long long n_rows,
                                                      long long* __restrict__ row_ptr) {
  const long long r = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (r > n_rows) return;
  const unsigned long long k = (unsigned long long)r << 32;
  long long lo = 0, hi = nnz;                            // first key >= k
  while (lo < hi) {
    const long long mid = (lo + hi) >> 1;
    if (keys[mid] < k) lo = mid + 1; else hi = mid;
  }
  row_ptr[r] = lo;
}

// one warp per row (same reductions as row_nnz_kernel: integer sums, so the order does not matter)
__global__ void __launch_bounds__(256) tally_stats_kernel(const unsigned long long* __restrict__ keys, const unsigned long long* __restrict__ vals,
                                                          const long long* __restrict__ row_ptr, int n_bins, int bin, int n_rows, int n_cols,
                                                          int n_surf, int row_first, int row_stride, int* __restrict__ nnz,
                                                          unsigned long long* __restrict__ rowsum, unsigned long long* __restrict__ cross) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= n_rows) return;
  const size_t rk = (size_t)row * n_bins + bin;
  const long long b = row_ptr[rk], e = row_ptr[rk + 1];
  const bool row_surf = row_first + row * row_stride < n_surf;
  int cnt = 0;
  unsigned long long s = 0, x = 0;
  for (long long p = b + lane; p < e; p += 32) {
    const int j = (int)(keys[p] & 0xffffffffull);
    if (j >= n_cols) continue;
    const unsigned long long v = vals[p];
    ++cnt; s += v;
    if ((j < n_surf) != row_surf) x += v;
  }
  for (int o = 16; o > 0; o >>= 1) {
    cnt += __shfl_down_sync(0xffffffffu, cnt, o); s += __shfl_down_sync(0xffffffffu, s, o); x += __shfl_down_sync(0xffffffffu, x, o);
  }
  if (lane == 0) { nnz[row] = cnt; rowsum[row] = s; if (cross) cross[row] = x; }
}

// columns ascend within a row, so the entries below a crop n_cols are a prefix of it
__global__ void __launch_bounds__(256) tally_fill_kernel(const unsigned long long* __restrict__ keys, const unsigned long long* __restrict__ vals,
                                                         const long long* __restrict__ row_ptr, int n_bins, int bin, int n_rows, int n_cols,
                                                         const long long* __restrict__ out_ptr, const unsigned long long* __restrict__ rowsum,
                                                         bool divide, int* __restrict__ cols, unsigned long long* __restrict__ cnt_out,
                                                         double* __restrict__ fvals) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= n_rows) return;
  const size_t rk = (size_t)row * n_bins + bin;
  const long long b = row_ptr[rk], e = row_ptr[rk + 1], o = out_ptr[row];
  const unsigned long long tot = rowsum[row];
  const double inv = tot ? 1.0 / (double)tot : 0.0;
  for (long long p = b + lane; p < e; p += 32) {
    const int j = (int)(keys[p] & 0xffffffffull);
    if (j >= n_cols) break;
    const unsigned long long v = vals[p];
    const long long k = o + (p - b);
    if (cols) cols[k] = j;
    if (cnt_out) cnt_out[k] = v;
    if (fvals) fvals[k] = divide ? (double)v / (double)tot : (double)v * inv;   // rthx_counts_csc : rthx_counts_csr
  }
}

template <class IDX>
__global__ void __launch_bounds__(256) key_index_kernel(const unsigned long long* __restrict__ keys, long long nnz, int base, IDX* __restrict__ out) {
  for (long long p = blockIdx.x * (long long)blockDim.x + threadIdx.x; p < nnz; p += (long long)gridDim.x * blockDim.x)
    out[p] = (IDX)(keys[p] & 0xffffffffull) + base;
}

unsigned flat_grid(long long n) { return (unsigned)std::max<long long>(1, std::min<long long>((n + 255) / 256, 148 * 32)); }

// Merge of two sorted key sets, each key at most once per set (rthx_trace_exchange_continue): merge path over the sequence of all
// na + nb keys, A before B on equal keys.  Thread t walks the MERGE_ITEMS positions from diagonal t * MERGE_ITEMS on.  A position that
// takes A[i] emits it plus B[j] when B[j] is the same key; a position that takes B[j] emits it unless A[i-1] was that key (then it was
// summed there).  Pass 1 counts the emitted keys per tile, pass 2 walks again, stages them in shared memory and writes them at the
// scanned tile offsets.
constexpr int MERGE_THREADS = 128, MERGE_ITEMS = 16, MERGE_TILE = MERGE_THREADS * MERGE_ITEMS;

__device__ __forceinline__ long long merge_split(const unsigned long long* __restrict__ a, long long na, const unsigned long long* __restrict__ b,
                                                 long long nb, long long d) {
  long long lo = d > nb ? d - nb : 0, hi = d < na ? d : na;   // A elements among the first d positions
  while (lo < hi) {
    const long long mid = (lo + hi) >> 1;
    if (a[mid] <= b[d - 1 - mid]) lo = mid + 1; else hi = mid;
  }
  return lo;
}

template <bool WRITE>
__device__ __forceinline__ int merge_walk(const unsigned long long* __restrict__ ak, const unsigned long long* __restrict__ av, long long na,
                                          const unsigned long long* __restrict__ bk, const unsigned long long* __restrict__ bv, long long nb,
                                          long long i, long long j, int steps, unsigned long long* __restrict__ ok,
                                          unsigned long long* __restrict__ ov, long long o) {
  int n = 0;
  for (int s = 0; s < steps; ++s) {
    if (i < na && (j >= nb || ak[i] <= bk[j])) {
      if (WRITE) {
        const unsigned long long k = ak[i];
        ok[o + n] = k;
        ov[o + n] = av[i] + (j < nb && bk[j] == k ? bv[j] : 0ull);
      }
      ++i; ++n;
    } else {
      const unsigned long long k = bk[j];
      if (i == 0 || ak[i - 1] != k) {
        if (WRITE) { ok[o + n] = k; ov[o + n] = bv[j]; }
        ++n;
      }
      ++j;
    }
  }
  return n;
}

template <bool WRITE>
__global__ void __launch_bounds__(MERGE_THREADS) tally_merge_kernel(const unsigned long long* __restrict__ ak, const unsigned long long* __restrict__ av,
                                                                    long long na, const unsigned long long* __restrict__ bk,
                                                                    const unsigned long long* __restrict__ bv, long long nb,
                                                                    long long* __restrict__ tile_cnt, const long long* __restrict__ tile_off,
                                                                    unsigned long long* __restrict__ ok, unsigned long long* __restrict__ ov) {
  using Scan = cub::BlockScan<int, MERGE_THREADS>;
  __shared__ typename Scan::TempStorage scan_tmp;
  const long long d = ((long long)blockIdx.x * MERGE_THREADS + threadIdx.x) * MERGE_ITEMS;
  const long long left = na + nb - d;
  const int steps = left <= 0 ? 0 : (left < MERGE_ITEMS ? (int)left : MERGE_ITEMS);
  long long i = 0, j = 0;
  int n = 0;
  if (steps > 0) {
    i = merge_split(ak, na, bk, nb, d); j = d - i;
    n = merge_walk<false>(ak, av, na, bk, bv, nb, i, j, steps, nullptr, nullptr, 0);
  }
  int off = 0, sum = 0;
  Scan(scan_tmp).ExclusiveSum(n, off, sum);
  if (!WRITE) {
    if (threadIdx.x == 0) tile_cnt[blockIdx.x] = sum;
    return;
  }
  if constexpr (WRITE) {
    // each thread's keys are consecutive, so direct stores would be strided across the warp: the tile is staged in shared memory
    // and written out with coalesced stores
    __shared__ unsigned long long s_k[MERGE_TILE], s_v[MERGE_TILE];
    if (steps > 0) merge_walk<true>(ak, av, na, bk, bv, nb, i, j, steps, s_k, s_v, off);
    __syncthreads();
    const long long base = tile_off[blockIdx.x];
    for (int t = threadIdx.x; t < sum; t += MERGE_THREADS) { ok[base + t] = s_k[t]; ov[base + t] = s_v[t]; }
  }
}
}  // namespace

long long tally_merge_tiles(long long n) { return (n + MERGE_TILE - 1) / MERGE_TILE; }

size_t tally_merge_temp_bytes(long long n_tiles) {
  size_t b = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, b, (const long long*)nullptr, (long long*)nullptr, (int)(n_tiles + 1));
  return b;
}

cudaError_t tally_merge(const unsigned long long* ak, const unsigned long long* av, long long na, const unsigned long long* bk,
                        const unsigned long long* bv, long long nb, unsigned long long* ok, unsigned long long* ov, long long* tiles,
                        void* temp, size_t temp_bytes, cudaStream_t st) {
  const long long n_tiles = tally_merge_tiles(na + nb);
  long long* cnt = tiles;
  long long* off = tiles + n_tiles + 1;
  cudaError_t e;
  if ((e = cudaMemsetAsync(cnt + n_tiles, 0, sizeof(long long), st)) != cudaSuccess) return e;
  if (n_tiles > 0) {
    tally_merge_kernel<false><<<(unsigned)n_tiles, MERGE_THREADS, 0, st>>>(ak, av, na, bk, bv, nb, cnt, nullptr, nullptr, nullptr);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
  }
  if ((e = cub::DeviceScan::ExclusiveSum(temp, temp_bytes, (const long long*)cnt, off, (int)(n_tiles + 1), st)) != cudaSuccess) return e;
  if (n_tiles > 0) tally_merge_kernel<true><<<(unsigned)n_tiles, MERGE_THREADS, 0, st>>>(ak, av, na, bk, bv, nb, nullptr, off, ok, ov);
  return cudaGetLastError();
}

size_t tally_temp_bytes(long long n_pairs) {
  const int n = (int)std::max<long long>(n_pairs, 1);
  size_t a = 0, b = 0;
  cub::DoubleBuffer<unsigned long long> kb(nullptr, nullptr);
  cub::DoubleBuffer<uint32_t> vb(nullptr, nullptr);
  cub::DeviceRadixSort::SortPairs(nullptr, a, kb, vb, n, 0, 64);
  auto vin = thrust::make_transform_iterator((const uint32_t*)nullptr, WidenU32());
  cub::DeviceReduce::ReduceByKey(nullptr, b, (const unsigned long long*)nullptr, (unsigned long long*)nullptr, vin, (unsigned long long*)nullptr,
                                 (long long*)nullptr, cuda::std::plus<unsigned long long>(), n);
  return std::max(a, b);
}

cudaError_t tally_reduce(unsigned long long* keys, uint32_t* cnt, unsigned long long* keys_alt, uint32_t* cnt_alt, long long n_pairs, int end_bit,
                         unsigned long long* out_keys, unsigned long long* out_vals, long long* n_unique_dev, void* temp, size_t temp_bytes,
                         cudaStream_t st) {
  cudaError_t e;
  if (n_pairs <= 0) return cudaMemsetAsync(n_unique_dev, 0, sizeof(long long), st);
  cub::DoubleBuffer<unsigned long long> kb(keys, keys_alt);
  cub::DoubleBuffer<uint32_t> vb(cnt, cnt_alt);
  if ((e = cub::DeviceRadixSort::SortPairs(temp, temp_bytes, kb, vb, (int)n_pairs, 0, end_bit, st)) != cudaSuccess) return e;
  auto vin = thrust::make_transform_iterator((const uint32_t*)vb.Current(), WidenU32());
  if ((e = cub::DeviceReduce::ReduceByKey(temp, temp_bytes, (const unsigned long long*)kb.Current(), out_keys, vin, out_vals, n_unique_dev,
                                          cuda::std::plus<unsigned long long>(), (int)n_pairs, st)) != cudaSuccess)
    return e;
  return cudaGetLastError();
}

cudaError_t tally_row_ptr(const unsigned long long* keys, long long nnz, long long n_rows, long long* row_ptr, cudaStream_t st) {
  row_ptr_kernel<<<(unsigned)((n_rows + 1 + 255) / 256), 256, 0, st>>>(keys, nnz, n_rows, row_ptr);
  return cudaGetLastError();
}

cudaError_t tally_row_stats(const unsigned long long* keys, const unsigned long long* vals, const long long* row_ptr, int n_bins, int bin, int n_rows,
                            int n_cols, int n_surf, int row_first, int row_stride, int* nnz, unsigned long long* rowsum, unsigned long long* cross,
                            cudaStream_t st) {
  if (n_rows > 0)
    tally_stats_kernel<<<(n_rows + 7) / 8, 256, 0, st>>>(keys, vals, row_ptr, n_bins, bin, n_rows, n_cols, n_surf, row_first, row_stride, nnz, rowsum, cross);
  return cudaGetLastError();
}

cudaError_t tally_row_fill(const unsigned long long* keys, const unsigned long long* vals, const long long* row_ptr, int n_bins, int bin, int n_rows,
                           int n_cols, const long long* out_ptr, const unsigned long long* rowsum, bool divide, int* cols, unsigned long long* cnt_out,
                           double* fvals, cudaStream_t st) {
  if (n_rows > 0)
    tally_fill_kernel<<<(n_rows + 7) / 8, 256, 0, st>>>(keys, vals, row_ptr, n_bins, bin, n_rows, n_cols, out_ptr, rowsum, divide, cols, cnt_out, fvals);
  return cudaGetLastError();
}

cudaError_t tally_key_index(const unsigned long long* keys_sorted, long long nnz, int base, void* out, bool i64, cudaStream_t st) {
  if (nnz <= 0) return cudaSuccess;
  if (i64) key_index_kernel<long long><<<flat_grid(nnz), 256, 0, st>>>(keys_sorted, nnz, base, (long long*)out);
  else key_index_kernel<int><<<flat_grid(nnz), 256, 0, st>>>(keys_sorted, nnz, base, (int*)out);
  return cudaGetLastError();
}

}  // namespace rthx
