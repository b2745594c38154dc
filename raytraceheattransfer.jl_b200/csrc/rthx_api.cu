// rthx_api.cu — host side of the C ABI in include/rthx.h: mesh preparation, device residency, launches, copies.
//
// Mesh preparation derives, once per rthx_create, everything the kernels need beyond the caller's arrays:
//   emitter table (createIndexMapping2D.jl:1-20), unit edge normals (calculateInwardNormal.jl:1-12),
//   reference-faithful locator grids (spatialAccelerations.jl:2-89), a coarse-face neighbour table (new) and,
//   where the fine cells of a coarse face are verified to be the affine lattice produced by meshQuad.jl:116-136 /
//   meshTriangle.jl:40-97, the analytic lattice inverse used instead of grid + point-in-polygon.
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "rthx_internal.h"
#include "rthx_grid.h"

using namespace rthx;

// Device resources that outlive a handle.  Callers re-create handles for every trace (the mesh is re-flattened on
// each call, like the reference re-reads its structs); creating/destroying streams, events and device allocations
// each time costs milliseconds on one GPU and >100 ms per cudaFree once peer mappings exist (NCCL / CUDA IPC).
// rthx_destroy therefore parks the bundle in a per-device pool and rthx_create adopts it; rthx_release_cached frees.
struct DevRes {
  cudaStream_t stream = nullptr;       // compute stream A (+ zeroing, recorder)
  cudaStream_t stream2 = nullptr;      // compute stream B: row batches alternate A/B so tails overlap
  cudaStream_t copy_stream = nullptr;  // device->host copies of finished row batches
  cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
  cudaEvent_t bev[18] = {};            // per-batch completion events (+2 scratch)
  void* arena = nullptr;                    size_t arena_cap = 0;      // mesh tables
  void* generic_arena = nullptr;            size_t generic_cap = 0;    // tables of the reference-faithful locator (built on first use)
  unsigned long long* counts_dev = nullptr; size_t counts_cap = 0;     // count matrix of the host-output entry points
  double* rec_pts_dev = nullptr;            size_t rec_pts_cap = 0;
  uint8_t* rec_valid_dev = nullptr;         size_t rec_valid_cap = 0;
  double* peak_dev = nullptr;
  int* csr_nnz = nullptr;                   size_t csr_cap = 0;        // per-row nnz (int), row totals, row pointers
  unsigned long long* csr_rowsum = nullptr; long long* csr_rowptr = nullptr; unsigned long long* csr_cross = nullptr;
  unsigned int* row_done_dev = nullptr;     size_t row_done_cap = 0;   // fused peer flush: per-row hand-over tickets
  int* csc_partial = nullptr;               size_t csc_partial_cap = 0; // CSC read-out: per (row tile, column) counts / offsets
  long long* csc_colptr = nullptr;          size_t csc_colptr_cap = 0;
  void* csr_out = nullptr;                  size_t csr_out_cap = 0;    // compacted cols / vals / F_vals
  double* smooth_X = nullptr;               size_t smooth_cap = 0;     // n*n doubles of the smoothing iterate
  double* smooth_vec = nullptr;             size_t smooth_vec_cap = 0; // w, rs, r, u, part (5 n doubles)
  void* smooth_src = nullptr;               size_t smooth_src_cap = 0; // staged host matrix (FROM_COUNTS / FROM_F)
  double* dyk_buf = nullptr;                size_t dyk_cap = 0;        // Dykstra rounds: Xbar / F iterate (+ second iterate and P for k > 1)
  // sparse smoothing (rthx_smooth_sparse): F as CSC and as sorted transpose keys, the CSR iterate X, work vectors, sort scratch
  long long* sp_ptr = nullptr;              size_t sp_ptr_cap = 0;     // colptr of F | row pointers of F | row pointers of X (3 (n+1))
  int* sp_rowval = nullptr;                 size_t sp_rowval_cap = 0;  // rowval of F
  double* sp_val = nullptr;                 size_t sp_val_cap = 0;     // values of F as CSC | in row order (2 nnz_F)
  unsigned long long* sp_keys = nullptr;    size_t sp_keys_cap = 0;    // transpose keys | sorted keys (2 nnz_F); index read-out scratch
  int* sp_xcol = nullptr;                   size_t sp_xcol_cap = 0;    // X / F_smooth: column indices
  double* sp_xval = nullptr;                size_t sp_xval_cap = 0;    // X / F_smooth: values
  double* sp_vec = nullptr;                 size_t sp_vec_cap = 0;     // w, r, u, u', part (5 n) + 8 scalars
  void* sp_tmp = nullptr;                   size_t sp_tmp_cap = 0;     // radix-sort scratch (bytes)
  // hashed row tally (rthx_trace_exchange_sparse): pair buffer (keys | alternate keys | counts | alternate counts, 24 bytes a pair),
  // control words, reduction scratch, and the resident counts as sorted unique keys, u64 totals and row pointers
  void* sk_pairs = nullptr;                 size_t sk_pairs_cap = 0;   // in pairs
  unsigned long long* sk_ctl = nullptr;     size_t sk_ctl_cap = 0;     // [0] pairs, [1] overflow, [2] flushes, [3] unique keys of a group
  void* sk_tmp = nullptr;                   size_t sk_tmp_cap = 0;     // bytes
  unsigned long long* sk_keys = nullptr;    size_t sk_keys_cap = 0;
  unsigned long long* sk_vals = nullptr;    size_t sk_vals_cap = 0;
  long long* sk_rowptr = nullptr;           size_t sk_rowptr_cap = 0;
  double* solve_buf = nullptr;              size_t solve_cap = 0;      // Krylov basis + work vectors + matvec partials
  double* solve_mat = nullptr;              size_t solve_mat_cap = 0;  // staged host F of rthx_solve_grey (dense padded / CSC)
  void* stage[2] = {nullptr, nullptr};      size_t stage_cap = 0;      // pinned staging for pageable destinations
  void* xfer[2] = {nullptr, nullptr};       size_t xfer_cap = 0;       // device staging of a copy helper (multi-link device->host copies)
  cudaEvent_t cev[2] = {nullptr, nullptr};
  bool valid = false;
};

namespace { struct HostImage; }

struct rthx_handle : DevRes {
  int device = 0;
  std::shared_ptr<HostImage> image;    // host image of the mesh tables (shared by the handles of one rthx_create_multi call)
  bool generic_ready = false;          // generic-locator tables uploaded (ensure_generic)
  std::vector<rthx_handle*> helpers;   // handles on OTHER devices whose PCIe links carry slices of large result copies (rthx_set_copy_helpers)
  cudaDeviceProp prop{};
  int n_coarse = 0, n_cells = 0, n_bands = 0, ns = 0, N = 0, n_affine = 0, n_bilinear = 0;
  bool queue_ok = false;       // every face has an analytic locator (affine or bilinear)
  bool queue_general = false;  // ... but some are bilinear or some interface has no unique neighbour: the general queue variant
  bool coarse_fits_smem = false;
  bool has_eps = false;
  bool single_quad = false;    // one parallelogram coarse face: SQ kernel
  CoarseDev face0{};
  bool fast_ok = false;        // every coarse face affine + complete neighbour table + descriptors fit in smem
  size_t mesh_bytes = 0;
  TraceParams base{};          // mesh pointers filled once
  int last_trace_bins = 0; size_t last_trace_rows = 0;    // resident counts: bins, rows per bin (N, or the rows of a shard)
  int last_rank = 0, last_world = 1;                      // ... row y of the resident matrix is element last_rank + y * last_world
  bool sparse_counts = false;                             // the resident counts are the hashed tally's (sk_*), not counts_dev
  long long sk_nnz = 0;                                   // ... its non-zeros over all traced bins
  // The one trace (of the contiguous ray-id range [ray_lo, ray_hi)) the resident counts are those of; rthx_trace_exchange_continue
  // extends it.  Valid while last_trace_bins > 0.
  int resident_kind = 0;                                  // RESIDENT_*
  uint64_t res_seed = 0; double res_nudge = 0.0; int res_mode = 0, res_locator = 0;
  std::vector<int32_t> res_bins;
  int64_t ray_lo = 0, ray_hi = 0;
  int smooth_n = 0; size_t smooth_ldx = 0;                // F_smooth resident in smooth_X after rthx_smooth_F (0: none)
  int sparse_n = 0; long long sparse_nnz = 0;             // sparse F_smooth resident in sp_* after rthx_smooth_sparse (0: none)
  int csr_bin = -1; long long csr_total = 0;              // bin whose row pointers are prepared on the device
  int csc_bin = -1;                                       // bin whose column pointers are prepared on the device
  double csr_chi = 0.0;                                   // surface-gas cross-coupling of that bin's row-normalised F
  // views into the arena
  unsigned long long* lost_dev = nullptr;   size_t lost_cap = 0;
  int32_t* bins_dev = nullptr;              size_t bins_cap = 0;
  int32_t* rec_slot_dev = nullptr;
  std::string err;
};

static thread_local std::string g_create_err;
static int ensure_generic(rthx_handle* h);
static void release_generic_cache();

namespace {
std::mutex g_pool_mu;
std::vector<DevRes> g_pool[64];
cudaDeviceProp g_prop[64];
bool g_prop_ok[64] = {};
bool g_kernels_configured[64] = {};   // cudaFuncSetAttribute(max dynamic smem) done for every kernel variant on this device

void devres_free(DevRes& r) {
  cudaFree(r.smooth_X); cudaFree(r.smooth_vec); cudaFree(r.smooth_src); cudaFree(r.solve_buf); cudaFree(r.solve_mat); cudaFree(r.dyk_buf);
  cudaFree(r.sk_pairs); cudaFree(r.sk_ctl); cudaFree(r.sk_tmp); cudaFree(r.sk_keys); cudaFree(r.sk_vals); cudaFree(r.sk_rowptr);
  cudaFree(r.sp_ptr); cudaFree(r.sp_rowval); cudaFree(r.sp_val); cudaFree(r.sp_keys); cudaFree(r.sp_xcol); cudaFree(r.sp_xval); cudaFree(r.sp_vec); cudaFree(r.sp_tmp);
  cudaFree(r.csr_nnz); cudaFree(r.csr_rowsum); cudaFree(r.csr_rowptr); cudaFree(r.csr_out); cudaFree(r.csr_cross); cudaFree(r.csc_partial); cudaFree(r.csc_colptr); cudaFree(r.row_done_dev);
  cudaFree(r.arena); cudaFree(r.generic_arena); cudaFree(r.counts_dev); cudaFree(r.rec_pts_dev); cudaFree(r.rec_valid_dev); cudaFree(r.peak_dev);
  for (auto& e : r.ev) if (e) cudaEventDestroy(e);
  for (auto& e : r.bev) if (e) cudaEventDestroy(e);
  for (auto& e : r.cev) if (e) cudaEventDestroy(e);
  for (auto& sp : r.stage) if (sp) cudaFreeHost(sp);
  for (auto& xp : r.xfer) if (xp) cudaFree(xp);
  if (r.stream) cudaStreamDestroy(r.stream);
  if (r.stream2) cudaStreamDestroy(r.stream2);
  if (r.copy_stream) cudaStreamDestroy(r.copy_stream);
  r = DevRes();
}

cudaError_t devres_create(DevRes& r) {
  cudaError_t e;
  if ((e = cudaStreamCreateWithFlags(&r.stream, cudaStreamNonBlocking)) != cudaSuccess) return e;
  if ((e = cudaStreamCreateWithFlags(&r.stream2, cudaStreamNonBlocking)) != cudaSuccess) return e;
  if ((e = cudaStreamCreateWithFlags(&r.copy_stream, cudaStreamNonBlocking)) != cudaSuccess) return e;
  for (auto& ev : r.ev) if ((e = cudaEventCreate(&ev)) != cudaSuccess) return e;
  for (auto& ev : r.bev) if ((e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming)) != cudaSuccess) return e;
  for (auto& ev : r.cev) if ((e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming)) != cudaSuccess) return e;
  r.valid = true;
  return cudaSuccess;
}
}  // namespace

static int fail(rthx_handle* h, int code, const std::string& msg) {
  if (h) h->err = msg; else g_create_err = msg;
  return code;
}
#define CU(h, call)                                                                                   \
  do {                                                                                                \
    cudaError_t e_ = (call);                                                                          \
    if (e_ != cudaSuccess)                                                                            \
      return fail(h, RTHX_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));             \
  } while (0)

// All mesh tables live in ONE device allocation filled by ONE host-to-device copy: with peer access enabled (NCCL
// processes) every cudaMalloc / cudaFree maps or unmaps the range on the peers and costs milliseconds.
struct Arena {
  std::vector<unsigned char> host;   // image of the uploaded tables
  size_t total = 0;                  // arena size including the device-only scratch regions behind the image
  template <class T>
  size_t add(const std::vector<T>& v, size_t min_elems = 1) {
    const size_t off = (host.size() + 255) & ~size_t(255);
    const size_t n = std::max(v.size(), min_elems);
    host.resize(off + n * sizeof(T), 0);
    if (!v.empty()) std::memcpy(host.data() + off, v.data(), v.size() * sizeof(T));
    total = host.size();
    return off;
  }
  // device-only region (cleared / written by the library before every use): no host bytes, nothing to copy.  Only valid after
  // the last add().
  template <class T>
  size_t scratch(size_t n_elems) {
    const size_t off = (total + 255) & ~size_t(255);
    total = off + std::max<size_t>(n_elems, 1) * sizeof(T);
    return off;
  }
};

// ---------------------------------------------------------------------------------------------------------------
// host-side mesh preparation
// ---------------------------------------------------------------------------------------------------------------
namespace {

bool close_pt(double ax, double ay, double bx, double by, double tol) { return std::fabs(ax - bx) <= tol && std::fabs(ay - by) <= tol; }

// Try to recognise the fine cells [f0, f0 + n_fine) of coarse face `cp` as the lattice of meshQuad / meshTriangle (affine for
// parallelograms and mirrored triangles, bilinear for general convex quadrilaterals).  The cells are read from the caller's
// arrays.  On success fills the lattice fields of `out` (+ the lattice->fine table for triangles) and returns true.
bool detect_affine(const Poly& cp, const rthx_mesh* m, int f0, int n_fine, CoarseDev& out, std::vector<int32_t>& lattice) {
  const int32_t* cnv = m->cell_nv + f0;
  const double* cvx = m->cell_vx + 4 * (size_t)f0;
  const double* cvy = m->cell_vy + 4 * (size_t)f0;
  double scale = 0;
  for (int i = 0; i < cp.n; ++i) scale = std::max(scale, std::max(std::fabs(cp.vx[i]), std::fabs(cp.vy[i])));
  const double ext = std::max(cp.bb[1] - cp.bb[0], cp.bb[3] - cp.bb[2]);
  const double tol = 1e-9 * std::max(ext, 1e-300);
  double qx[4], qy[4];
  int Nx = 0, Ny = 0, mirror = -1, diag = -1;
  bool bilinear = false;
  if (cp.n == 4) {
    for (int i = 0; i < 4; ++i) { qx[i] = cp.vx[i]; qy[i] = cp.vy[i]; }
    if (!close_pt(qx[0] - qx[1] + qx[2] - qx[3], qy[0] - qy[1] + qy[2] - qy[3], 0, 0, 1e-12 * std::max(scale, ext))) {
      // no parallelogram: meshQuad.jl:116-136 still produces a structured lattice — the bilinear image of the unit square.
      // Accept strictly convex CCW quadrilaterals (the inverse map below is single-valued on them).
      for (int i = 0; i < 4; ++i) {
        const int j = (i + 1) & 3, k = (i + 2) & 3;
        const double cr = (qx[j] - qx[i]) * (qy[k] - qy[j]) - (qy[j] - qy[i]) * (qx[k] - qx[j]);
        if (!(cr > 1e-9 * ext * ext)) return false;
      }
      bilinear = true;
    }
    if (cnv[0] != 4) return false;
    const double e0 = std::hypot(cvx[1] - cvx[0], cvy[1] - cvy[0]);
    const double ab = std::hypot(qx[1] - qx[0], qy[1] - qy[0]);
    if (!(e0 > 0)) return false;
    Nx = (int)std::llround(ab / e0);
    if (Nx < 1 || n_fine % Nx != 0) return false;
    Ny = n_fine / Nx;
  } else {
    // meshTriangle.jl:15-53: longest edge (first maximum) is the cut diagonal, opposite vertex point-mirrored
    const double l0 = std::hypot(cp.vx[0] - cp.vx[1], cp.vy[0] - cp.vy[1]);
    const double l1 = std::hypot(cp.vx[1] - cp.vx[2], cp.vy[1] - cp.vy[2]);
    const double l2 = std::hypot(cp.vx[2] - cp.vx[0], cp.vy[2] - cp.vy[0]);
    int mi = 0;
    if (l1 > l0) mi = 1;
    if (l2 > std::max(l0, l1)) mi = 2;
    const int a = mi, b = (mi + 1) % 3, o = (mi + 2) % 3;  // edge a->b is the diagonal, o the opposite vertex
    const double mx = cp.vx[a] + (cp.vx[b] - cp.vx[a]) / 2, my = cp.vy[a] + (cp.vy[b] - cp.vy[a]) / 2;
    const double rx = -(cp.vx[o] - mx) + mx, ry = -(cp.vy[o] - my) + my;
    // new_points: mirrored vertex inserted after the start of the longest edge
    int w = 0;
    for (int i = 0; i < 3; ++i) {
      qx[w] = cp.vx[i]; qy[w] = cp.vy[i]; ++w;
      if (i == mi) { qx[w] = rx; qy[w] = ry; mirror = w; ++w; }
    }
    diag = mi;
    const long long nd = (long long)std::llround((std::sqrt(8.0 * n_fine + 1.0) - 1.0) / 2.0);
    if (nd < 1 || nd * (nd + 1) / 2 != n_fine) return false;
    Nx = Ny = (int)nd;
  }
  // lattice vertex (n,m) of the map  A + s (B-A) + t (D-A) + s t (A-B+C-D),  s = n/Nx, t = m/Ny  (the last term vanishes for
  // parallelograms and mirrored triangles: affine)
  const double Gx = bilinear ? qx[0] - qx[1] + qx[2] - qx[3] : 0.0, Gy = bilinear ? qy[0] - qy[1] + qy[2] - qy[3] : 0.0;
  auto lat = [&](int n, int m_, double& x, double& y) {
    const double s = (double)n / Nx, t = (double)m_ / Ny;
    x = qx[0] + s * (qx[1] - qx[0]) + t * (qx[3] - qx[0]) + s * t * Gx;
    y = qy[0] + s * (qy[1] - qy[0]) + t * (qy[3] - qy[0]) + s * t * Gy;
  };
  std::vector<int32_t> table;
  if (cp.n == 3) table.assign((size_t)Nx * Ny, -1);
  int idx = 0;
  for (int mm = 0; mm < Ny; ++mm)
    for (int n = 0; n < Nx; ++n) {
      double lx[4], ly[4];
      lat(n, mm, lx[0], ly[0]); lat(n + 1, mm, lx[1], ly[1]); lat(n + 1, mm + 1, lx[2], ly[2]); lat(n, mm + 1, lx[3], ly[3]);
      if (idx < n_fine) {
        const int cn = cnv[idx];
        const double* x = cvx + 4 * (size_t)idx;
        const double* y = cvy + 4 * (size_t)idx;
        bool match = false;
        if (cn == 4) {
          match = true;
          for (int i = 0; i < 4; ++i) match = match && close_pt(x[i], y[i], lx[i], ly[i], tol);
        } else if (cp.n == 3) {
          // diagonal cell: the three lattice corners other than the mirrored one (meshTriangle.jl:55,83)
          match = true;
          int w = 0;
          for (int i = 0; i < 4; ++i) {
            if (i == mirror) continue;
            match = match && close_pt(x[w], y[w], lx[i], ly[i], tol);
            ++w;
          }
        }
        if (match) {
          if (cp.n == 3) table[(size_t)n + (size_t)mm * Nx] = idx;
          ++idx;
          continue;
        }
      }
      if (cp.n == 4) return false;  // every lattice cell of a quad must be present, in order
    }
  if (idx != n_fine) return false;
  // inverse map: [s;t] = diag(Nx,Ny) * inv([B-A, D-A]) * (p - A)
  const double ux = qx[1] - qx[0], uy = qy[1] - qy[0], vx = qx[3] - qx[0], vy = qy[3] - qy[0];
  const double det = ux * vy - uy * vx;
  if (!(std::fabs(det) > 0)) return false;
  out.ax = qx[0]; out.ay = qy[0];
  if (bilinear) {
    // device: a2 s^2 + a1 s + a0 = 0 with a2 = E x G, a1 = E x F - H x G, a0 = -H x F (H = p - A); t by projection on F + s G
    out.g1x = ux; out.g1y = uy; out.g2x = vx; out.g2y = vy;
    out.cen[0] = Gx; out.cen[1] = Gy;
    const double a2 = ux * Gy - uy * Gx;
    out.hw[0] = a2 != 0.0 ? 1.0 / a2 : INFINITY;
    out.hw[1] = det;
    out.Nx = Nx; out.Ny = Ny;
    out.kind = KIND_BILINEAR_QUAD; out.lat_off = -1; out.diag = -1;
    return true;
  }
  out.g1x = Nx * (vy / det);  out.g1y = Nx * (-vx / det);
  out.g2x = Ny * (-uy / det); out.g2y = Ny * (ux / det);
  out.Nx = Nx; out.Ny = Ny;
  if (cp.n == 4) { out.kind = KIND_AFFINE_QUAD; out.lat_off = -1; out.diag = -1; }
  else {
    out.kind = KIND_AFFINE_TRI; out.diag = diag;
    out.lat_off = (int32_t)lattice.size();
    lattice.insert(lattice.end(), table.begin(), table.end());
  }
  return true;
}

// Page-locked host buffers for mesh images, pooled per process: callers re-create the handle for every trace, and a
// cudaHostAlloc / cudaFreeHost pair costs far more than the mesh preparation itself.
std::mutex g_pin_mu;
std::vector<std::pair<unsigned char*, size_t>> g_pin_pool;

unsigned char* take_pinned(size_t bytes, size_t* cap) {
  {
    std::lock_guard<std::mutex> lk(g_pin_mu);
    for (size_t i = 0; i < g_pin_pool.size(); ++i)
      if (g_pin_pool[i].second >= bytes) {
        unsigned char* p = g_pin_pool[i].first; *cap = g_pin_pool[i].second;
        g_pin_pool.erase(g_pin_pool.begin() + (long)i);
        return p;
      }
  }
  void* p = nullptr;
  const size_t want = bytes + bytes / 4 + 4096;
#ifdef RTHX_PREP_BENCH   // tools/hostbench/prep_bench.cu: times the host preparation on a machine without a GPU
  p = std::malloc(want);
  if (!p) return nullptr;
#else
  if (cudaHostAlloc(&p, want, cudaHostAllocPortable) != cudaSuccess) { cudaGetLastError(); return nullptr; }
#endif
  *cap = want;
  return static_cast<unsigned char*>(p);
}
void give_pinned(unsigned char* p, size_t cap) {
  if (!p) return;
  std::lock_guard<std::mutex> lk(g_pin_mu);
  if (g_pin_pool.size() < 8) { g_pin_pool.emplace_back(p, cap); return; }
  cudaFreeHost(p);
}

// Everything rthx_create derives from the caller's arrays, as ONE image of the device arena in page-locked host memory, plus
// the block-uniform facts the launch planner needs.  Built once per rthx_create / rthx_create_multi call and shared by the
// handles created from it (the generic-locator tables are derived from it on first use).
struct HostImage {
  unsigned char* data = nullptr;
  size_t cap = 0, bytes = 0, total = 0;      // pinned capacity, image bytes, arena bytes incl. the device-only scratch regions
  size_t o_coarse = 0, o_sets = 0, o_bent = 0, o_bcand = 0, o_frec = 0, o_nv = 0, o_pvx = 0, o_pvy = 0, o_mid = 0, o_vol = 0, o_surf = 0, o_beta = 0,
         o_ub = 0, o_lat = 0, o_abs = 0, o_omega = 0, o_omu = 0, o_eps = 0, o_ec = 0, o_ew = 0, o_eco = 0, o_bins = 0, o_rec = 0, o_lost = 0;
  int nc = 0, ncell = 0, ns = 0, N = 0, nb = 0, n_affine = 0, n_bilinear = 0;
  bool has_eps = false, nbr_complete = true, needs_generic = false;
  CoarseDev face0{};
  std::vector<Poly> coarse_polys;
  std::vector<int32_t> fine_off;
  ~HostImage() { give_pinned(data, cap); }
  template <class T> T* at(size_t off) const { return reinterpret_cast<T*>(data + off); }
};

struct Layout {            // running offset of the arena image: every table 256-byte aligned
  size_t total = 0;
  size_t add(size_t bytes) { const size_t off = (total + 255) & ~size_t(255); total = off + std::max<size_t>(bytes, 8); return off; }
};

// Host-only half of rthx_create.  Returns RTHX_OK and the image, or an error code with the message in `err`.
int prepare_mesh(const rthx_mesh* m, std::shared_ptr<HostImage>& out, std::string& err) {
  const bool timing = std::getenv("RTHX_CREATE_TIMING") != nullptr;
  auto t_prev = std::chrono::steady_clock::now();
  auto lap = [&](const char* what) {
    if (!timing) return;
    const auto t = std::chrono::steady_clock::now();
    std::fprintf(stderr, "rthx_create: %-28s %8.3f ms\n", what, std::chrono::duration<double, std::milli>(t - t_prev).count());
    t_prev = t;
  };
  auto im = std::make_shared<HostImage>();
  const int nc = m->n_coarse, ncell = m->n_cells, ns = m->n_surfaces, N = ns + ncell, nb = m->n_bands;
  im->nc = nc; im->ncell = ncell; im->ns = ns; im->N = N; im->nb = nb;
  if (m->fine_off[0] != 0 || m->fine_off[nc] != ncell) { err = "rthx_create: fine_off must span [0, n_cells]"; return RTHX_ERR_ARG; }
  for (int g = 0; g < ncell; ++g)
    if (m->cell_nv[g] != 3 && m->cell_nv[g] != 4) { err = "rthx_create: cell_nv must be 3 or 4"; return RTHX_ERR_ARG; }
  im->fine_off.assign(m->fine_off, m->fine_off + nc + 1);
  // coarse polygons (normals, bounding boxes); the fine cells get theirs only if the generic locator is ever needed
  std::vector<Poly>& cpolys = im->coarse_polys;
  cpolys.resize(nc);
  for (int c = 0; c < nc; ++c) {
    Poly& p = cpolys[c];
    p.n = m->coarse_nv[c];
    if (p.n != 3 && p.n != 4) { err = "rthx_create: coarse_nv must be 3 or 4"; return RTHX_ERR_ARG; }
    double sx = 0, sy = 0;
    for (int i = 0; i < p.n; ++i) { p.vx[i] = m->coarse_vx[4 * c + i]; p.vy[i] = m->coarse_vy[4 * c + i]; sx += p.vx[i]; sy += p.vy[i]; }
    p.midx = sx / p.n; p.midy = sy / p.n;
    if (p.n == 4)
      p.volume = 0.5 * (p.vx[0] * (p.vy[1] - p.vy[2]) + p.vx[1] * (p.vy[2] - p.vy[0]) + p.vx[2] * (p.vy[0] - p.vy[1])) +
                 0.5 * (p.vx[2] * (p.vy[3] - p.vy[0]) + p.vx[3] * (p.vy[0] - p.vy[2]) + p.vx[0] * (p.vy[2] - p.vy[3]));
    else
      p.volume = 0.5 * (p.vx[0] * (p.vy[1] - p.vy[2]) + p.vx[1] * (p.vy[2] - p.vy[0]) + p.vx[2] * (p.vy[0] - p.vy[1]));
    poly_finish(p);
    if (m->fine_off[c + 1] <= m->fine_off[c]) { err = "rthx_create: every coarse face needs at least one fine cell"; return RTHX_ERR_ARG; }
  }
  lap("coarse polygons");

  // coarse descriptors: lattice detection, absorber tables, neighbour table; the coarse-set locator grid (set 0)
  std::vector<FaceSetDev> sets(1 + (size_t)nc);
  std::memset(sets.data(), 0, sizeof(FaceSetDev) * sets.size());
  std::vector<int32_t> bent, bcand, lattice, abs_tab;
  build_grid(cpolys.data(), nc, ncell, sets[0], bent, bcand);  // set 0 (coarse faces) only; the fine sets belong to ensure_generic
  std::vector<CoarseDev> coarse(nc);
  const double ext_tol = 1e-9;
  for (int c = 0; c < nc; ++c) {
    const Poly& cp = cpolys[c];
    const int f0 = m->fine_off[c], nf = m->fine_off[c + 1] - f0;
    CoarseDev& d = coarse[c];
    std::memset(&d, 0, sizeof(d));
    for (int i = 0; i < 4; ++i) { d.vx[i] = cp.vx[i]; d.vy[i] = cp.vy[i]; d.nx[i] = cp.nx[i]; d.ny[i] = cp.ny[i]; d.nbr[i] = -1; d.solid[i] = 0; }
    for (int i = 0; i < cp.n; ++i) d.solid[i] = m->coarse_solid[4 * c + i] ? 1 : 0;
    d.nv = cp.n; d.fine_off = f0; d.kind = KIND_GENERIC; d.lat_off = -1; d.diag = -1; d.Nx = d.Ny = 0;
    if (detect_affine(cp, m, f0, nf, d, lattice)) { if (d.kind == KIND_BILINEAR_QUAD) im->n_bilinear++; else im->n_affine++; }
    for (int i = 0; i < cp.n; ++i) d.h[i] = cp.vx[i] * cp.nx[i] + cp.vy[i] * cp.ny[i];
    if (d.kind == KIND_AFFINE_QUAD) {   // slab form: opposite edges measured along the normals of edges 0 and 1
      d.h[2] = cp.vx[2] * cp.nx[0] + cp.vy[2] * cp.ny[0];
      d.h[3] = cp.vx[3] * cp.nx[1] + cp.vy[3] * cp.ny[1];
      d.cen[0] = 0.5 * (d.h[0] + d.h[2]); d.hw[0] = 0.5 * (d.h[0] - d.h[2]);
      d.cen[1] = 0.5 * (d.h[1] + d.h[3]); d.hw[1] = 0.5 * (d.h[1] - d.h[3]);
    }
    // Absorber table of an affine face: for every lattice cell the element a ray ending there is tallied in — entry 0 for a gas
    // event (Ns + global cell index, getGlobalIndex2D.jl:10), entry 1+k for a hit on coarse edge k: the surface index of the fine
    // wall lying on that edge (fine wall = k, except in the quad cells of a mirrored-triangle lattice, whose walls are numbered
    // around the uncut parallelogram: the cut diagonal is no wall of theirs and the walls behind it shift by one), -1 where the
    // fine wall is not solid or the lattice cell lies outside the triangle.
    d.abs_off = -1;
    if (d.kind != KIND_GENERIC) {
      d.abs_off = (int32_t)(abs_tab.size() / 5);
      const size_t ncell_lat = (size_t)d.Nx * d.Ny;
      const size_t base = abs_tab.size();
      abs_tab.resize(base + 5 * ncell_lat, -1);
      for (size_t l = 0; l < ncell_lat; ++l) {
        const int f = d.kind == KIND_AFFINE_TRI ? lattice[(size_t)d.lat_off + l] : (int)l;   // quad lattices (affine or bilinear): fine index = n + m Nx
        if (f < 0) continue;
        int32_t* row = abs_tab.data() + base + 5 * l;
        const int gc = f0 + f;
        row[0] = ns + gc;
        for (int k = 0; k < cp.n; ++k) {
          int w = k;
          if (d.kind == KIND_AFFINE_TRI && m->cell_nv[gc] != 3) {
            if (k == d.diag) continue;
            w = k < d.diag ? k : k + 1;
          }
          row[1 + k] = m->cell_surf_id[4 * (size_t)gc + w];
        }
      }
    } else {
      im->needs_generic = true;
    }
  }
  lap("lattice detection + tables");
  // neighbour table: the unique coarse face sharing the (reversed) edge; T-junctions stay -1 (generic search)
  for (int c = 0; c < nc; ++c) {
    const Poly& a = cpolys[c];
    const double tol = ext_tol * std::max(a.bb[1] - a.bb[0], a.bb[3] - a.bb[2]);
    for (int k = 0; k < a.n; ++k) {
      if (coarse[c].solid[k]) continue;
      const int k2 = (k + 1) % a.n;
      int found = -1, n_found = 0;
      for (int c2 = 0; c2 < nc; ++c2) {
        if (c2 == c) continue;
        const Poly& b = cpolys[c2];
        for (int j = 0; j < b.n; ++j) {
          const int j2 = (j + 1) % b.n;
          if (close_pt(a.vx[k], a.vy[k], b.vx[j2], b.vy[j2], tol) && close_pt(a.vx[k2], a.vy[k2], b.vx[j], b.vy[j], tol)) { found = c2; ++n_found; }
        }
      }
      coarse[c].nbr[k] = (n_found == 1) ? found : -1;
      if (coarse[c].nbr[k] < 0) im->nbr_complete = false;   // open / T-junction edge: needs the coarse point location
    }
  }
  if (sizeof(CoarseDev) * (size_t)nc > 96 * 1024) im->needs_generic = true;   // > 384 coarse faces: read through L1/L2 by the generic kernel
  if (lattice.empty()) lattice.push_back(-1);
  if (abs_tab.empty()) abs_tab.assign(5, -1);
  im->face0 = coarse[0];
  im->has_eps = m->epsilon != nullptr || ns == 0;
  lap("neighbour table");

  // layout of the image, then fill it in place (page-locked: the H2D copies of several devices run concurrently by DMA)
  const size_t npoly = (size_t)ncell + nc;
  Layout L;
  im->o_coarse = L.add(sizeof(CoarseDev) * coarse.size()); im->o_sets = L.add(sizeof(FaceSetDev) * sets.size());
  im->o_bent = L.add(4 * bent.size()); im->o_bcand = L.add(4 * bcand.size()); im->o_frec = L.add(8 * FREC * (size_t)nc);
  im->o_nv = L.add(4 * npoly); im->o_pvx = L.add(32 * npoly); im->o_pvy = L.add(32 * npoly);
  im->o_mid = L.add(16 * (size_t)ncell); im->o_vol = L.add(8 * (size_t)ncell); im->o_surf = L.add(16 * (size_t)ncell);
  im->o_beta = L.add(8 * (size_t)nb * ncell); im->o_ub = L.add(8 * (size_t)nb);
  im->o_lat = L.add(4 * lattice.size()); im->o_abs = L.add(4 * abs_tab.size());
  im->o_omega = L.add(8 * (size_t)nb * ncell); im->o_omu = L.add(16 * (size_t)nb); im->o_eps = L.add(m->epsilon ? 8 * (size_t)nb * ns : 0);
  im->o_ec = L.add(4 * (size_t)N); im->o_ew = L.add(4 * (size_t)N); im->o_eco = L.add(4 * (size_t)N);
  im->bytes = L.total;
  im->o_bins = L.add(4 * ((size_t)nb * 4 + 16)); im->o_rec = L.add(4 * (size_t)N);
  im->o_lost = L.add(8 * ((size_t)nb * 4 + 16) * (size_t)N);
  im->total = L.total;
  im->data = take_pinned(im->bytes, &im->cap);
  if (!im->data) { err = "rthx_create: cudaHostAlloc(mesh image) failed"; return RTHX_ERR_NOMEM; }
  lap("pinned image");
  std::memcpy(im->at<CoarseDev>(im->o_coarse), coarse.data(), sizeof(CoarseDev) * coarse.size());
  std::memcpy(im->at<FaceSetDev>(im->o_sets), sets.data(), sizeof(FaceSetDev) * sets.size());
  std::memcpy(im->at<int32_t>(im->o_bent), bent.data(), 4 * bent.size());
  if (!bcand.empty()) std::memcpy(im->at<int32_t>(im->o_bcand), bcand.data(), 4 * bcand.size());
  for (int c = 0; c < nc; ++c) face_record(cpolys[c], nullptr, im->at<double>(im->o_frec) + FREC * (size_t)c);
  std::memcpy(im->at<int32_t>(im->o_lat), lattice.data(), 4 * lattice.size());
  std::memcpy(im->at<int32_t>(im->o_abs), abs_tab.data(), 4 * abs_tab.size());
  {
    int32_t* nv = im->at<int32_t>(im->o_nv);
    double* pvx = im->at<double>(im->o_pvx);
    double* pvy = im->at<double>(im->o_pvy);
    std::memcpy(nv, m->cell_nv, 4 * (size_t)ncell);
    std::memcpy(pvx, m->cell_vx, 32 * (size_t)ncell);
    std::memcpy(pvy, m->cell_vy, 32 * (size_t)ncell);
    for (int g = 0; g < ncell; ++g) if (nv[g] == 3) { pvx[4 * (size_t)g + 3] = 0.0; pvy[4 * (size_t)g + 3] = 0.0; }   // unused 4th slot: any value on input
    for (int c = 0; c < nc; ++c) {
      nv[ncell + c] = cpolys[c].n;
      for (int k = 0; k < 4; ++k) { pvx[4 * ((size_t)ncell + c) + k] = cpolys[c].vx[k]; pvy[4 * ((size_t)ncell + c) + k] = cpolys[c].vy[k]; }
    }
  }
  std::memcpy(im->at<double>(im->o_mid), m->cell_mid, 16 * (size_t)ncell);
  std::memcpy(im->at<double>(im->o_vol), m->cell_volume, 8 * (size_t)ncell);
  std::memcpy(im->at<int32_t>(im->o_surf), m->cell_surf_id, 16 * (size_t)ncell);
  std::memcpy(im->at<double>(im->o_ub), m->uniform_beta, 8 * (size_t)nb);
  {
    // beta = kappa + sigma_s; MULTI_BOUNCE properties: scattering albedo per (band, cell) — 0 where beta = 0 — and emissivity
    double* beta = im->at<double>(im->o_beta);
    double* omega = im->at<double>(im->o_omega);
    const size_t n = (size_t)nb * ncell;
    for (size_t i = 0; i < n; ++i) { const double b = m->kappa[i] + m->sigma_s[i]; beta[i] = b; omega[i] = b > 0.0 ? m->sigma_s[i] / b : 0.0; }
    double* band_u = im->at<double>(im->o_omu);            // a band whose cells share one albedo / whose walls share one emissivity:
    for (int b = 0; b < nb; ++b) {                         // the kernels read it once per block instead of once per event
      const double* ob = omega + (size_t)b * ncell;
      bool same = ncell > 0;
      for (int i = 1; i < ncell && same; ++i) same = ob[i] == ob[0];
      band_u[2 * b] = same ? ob[0] : -1.0;
      const double* eb = m->epsilon ? m->epsilon + (size_t)b * ns : nullptr;
      same = eb != nullptr && ns > 0;
      for (int i = 1; i < ns && same; ++i) same = eb[i] == eb[0];
      band_u[2 * b + 1] = same ? eb[0] : -1.0;
    }
    if (m->epsilon) std::memcpy(im->at<double>(im->o_eps), m->epsilon, 8 * (size_t)nb * ns);
  }
  {
    // emitter table in global-index order (createIndexMapping2D.jl:1-20): surfaces 0..Ns-1, then Ns + cell
    int32_t* em_cell = im->at<int32_t>(im->o_ec);
    int32_t* em_wall = im->at<int32_t>(im->o_ew);
    int32_t* em_coarse = im->at<int32_t>(im->o_eco);
    for (int s = 0; s < ns; ++s) em_cell[s] = -1;
    for (int c = 0; c < nc; ++c)
      for (int g = m->fine_off[c]; g < m->fine_off[c + 1]; ++g) {
        em_cell[ns + g] = g; em_wall[ns + g] = -1; em_coarse[ns + g] = c;
        const int n = m->cell_nv[g];
        for (int w = 0; w < n; ++w) {
          const int s = m->cell_surf_id[4 * (size_t)g + w];
          if (s < 0) continue;
          if (s >= ns || em_cell[s] != -1) { err = "rthx_create: cell_surf_id is not a permutation of 0..Ns-1"; return RTHX_ERR_ARG; }
          em_cell[s] = g; em_wall[s] = w; em_coarse[s] = c;
        }
      }
    for (int s = 0; s < ns; ++s) if (em_cell[s] < 0) { err = "rthx_create: surface index without a wall"; return RTHX_ERR_ARG; }
  }
  lap("image fill");
  out = im;
  return RTHX_OK;
}

}  // namespace

// ---------------------------------------------------------------------------------------------------------------
// create / destroy / info
// ---------------------------------------------------------------------------------------------------------------
extern "C" int rthx_version(void) { return RTHX_VERSION_MAJOR * 100 + RTHX_VERSION_MINOR; }

extern "C" const char* rthx_last_error(const rthx_handle* h) { return h ? h->err.c_str() : g_create_err.c_str(); }

extern "C" int rthx_destroy(rthx_handle* h) {
  if (!h) return RTHX_OK;
  cudaSetDevice(h->device);
  if (h->valid) {
    // drain this handle's streams, then park the resources for the next handle on this device
    cudaStreamSynchronize(h->stream); cudaStreamSynchronize(h->stream2); cudaStreamSynchronize(h->copy_stream);
    std::lock_guard<std::mutex> lk(g_pool_mu);
    g_pool[h->device & 63].push_back(static_cast<DevRes&>(*h));
  }
  delete h;
  return RTHX_OK;
}

extern "C" int rthx_release_cached(void) {
  std::lock_guard<std::mutex> lk(g_pool_mu);
  int cur = 0;
  cudaGetDevice(&cur);
  for (int d = 0; d < 64; ++d) {
    if (g_pool[d].empty()) continue;
    cudaSetDevice(d);
    for (auto& r : g_pool[d]) devres_free(r);
    g_pool[d].clear();
  }
  cudaSetDevice(cur);
  {
    std::lock_guard<std::mutex> lk2(g_pin_mu);
    for (auto& pb : g_pin_pool) cudaFreeHost(pb.first);
    g_pin_pool.clear();
  }
  release_generic_cache();
  return RTHX_OK;
}

namespace {

// Device half of rthx_create: adopt pooled resources, upload the image (asynchronously on the handle's stream), wire the
// table pointers.  `sync` waits for the upload; rthx_create_multi enqueues every device first and waits once.
int create_on_device(rthx_handle** out, const std::shared_ptr<HostImage>& im, int device_id, int n_dev, bool sync) {
  *out = nullptr;
  if (device_id < 0 || device_id >= n_dev) return fail(nullptr, RTHX_ERR_ARG, "rthx_create: bad device id");
  rthx_handle* h = new rthx_handle();
  h->device = device_id;
  cudaError_t ce;
  auto bail = [&](int code, const std::string& msg) { g_create_err = msg; rthx_destroy(h); return code; };
  if ((ce = cudaSetDevice(device_id)) != cudaSuccess) return bail(RTHX_ERR_CUDA, cudaGetErrorString(ce));
  {
    std::lock_guard<std::mutex> lk(g_pool_mu);
    if (!g_prop_ok[device_id & 63]) {
      if ((ce = cudaGetDeviceProperties(&g_prop[device_id & 63], device_id)) != cudaSuccess) { g_create_err = cudaGetErrorString(ce); delete h; return RTHX_ERR_CUDA; }
      g_prop_ok[device_id & 63] = true;
    }
    h->prop = g_prop[device_id & 63];
    auto& pool = g_pool[device_id & 63];
    if (!pool.empty()) { static_cast<DevRes&>(*h) = pool.back(); pool.pop_back(); }
  }
  if (h->prop.major < 10) return bail(RTHX_ERR_CUDA, "rthx_create: device is not sm_100 class (kernels are built for sm_100a only)");
  if (!h->valid && (ce = devres_create(*h)) != cudaSuccess) return bail(RTHX_ERR_CUDA, std::string("stream/event creation: ") + cudaGetErrorString(ce));
  h->image = im;
  h->n_coarse = im->nc; h->n_cells = im->ncell; h->ns = im->ns; h->N = im->N; h->n_bands = im->nb;
  h->n_affine = im->n_affine; h->n_bilinear = im->n_bilinear; h->has_eps = im->has_eps;
  if (h->arena_cap < im->total) {
    cudaFree(h->arena);
    h->arena = nullptr; h->arena_cap = 0;
    const size_t cap = im->total + im->total / 4;
    if ((ce = cudaMalloc(&h->arena, cap)) != cudaSuccess) return bail(RTHX_ERR_CUDA, std::string("cudaMalloc(mesh arena): ") + cudaGetErrorString(ce));
    h->arena_cap = cap;
  }
  if ((ce = cudaMemcpyAsync(h->arena, im->data, im->bytes, cudaMemcpyHostToDevice, h->stream)) != cudaSuccess)
    return bail(RTHX_ERR_CUDA, std::string("cudaMemcpyAsync(mesh arena): ") + cudaGetErrorString(ce));
  h->mesh_bytes = im->bytes;
  TraceParams& P = h->base;
  std::memset(&P, 0, sizeof(P));
  unsigned char* b8 = static_cast<unsigned char*>(h->arena);
  P.coarse = (const CoarseDev*)(b8 + im->o_coarse); P.sets = (const FaceSetDev*)(b8 + im->o_sets);
  // bucket grid + polygon records of the coarse set only (the general queue variant's crossing search; records are indexed by
  // polygon = n_cells + coarse face, so the base pointer is offset and never dereferenced below n_cells); ensure_generic re-points them
  P.bucket_ent = (const int4*)(b8 + im->o_bent); P.bucket_cand = (const int32_t*)(b8 + im->o_bcand);
  P.face_rec = (const double*)(b8 + im->o_frec) - FREC * (size_t)im->ncell;
  P.poly_nv = (const int32_t*)(b8 + im->o_nv); P.poly_vx = (const double*)(b8 + im->o_pvx); P.poly_vy = (const double*)(b8 + im->o_pvy);
  P.poly_nx = nullptr; P.poly_ny = nullptr;      // per-polygon normals belong to the generic tables (ensure_generic)
  P.cell_mid = (const double*)(b8 + im->o_mid); P.cell_volume = (const double*)(b8 + im->o_vol);
  P.cell_surf_id = (const int32_t*)(b8 + im->o_surf); P.beta = (const double*)(b8 + im->o_beta); P.uniform_beta = (const double*)(b8 + im->o_ub);
  P.omega = (const double*)(b8 + im->o_omega); P.band_u = (const double*)(b8 + im->o_omu); P.eps = (const double*)(b8 + im->o_eps);
  P.lattice = (const int32_t*)(b8 + im->o_lat); P.abs_tab = (const int32_t*)(b8 + im->o_abs);
  P.em_cell = (const int32_t*)(b8 + im->o_ec); P.em_wall = (const int32_t*)(b8 + im->o_ew); P.em_coarse = (const int32_t*)(b8 + im->o_eco);
  h->bins_dev = (int32_t*)(b8 + im->o_bins); h->bins_cap = (size_t)im->nb * 4 + 16;
  h->rec_slot_dev = (int32_t*)(b8 + im->o_rec);
  h->lost_dev = (unsigned long long*)(b8 + im->o_lost); h->lost_cap = ((size_t)im->nb * 4 + 16) * (size_t)im->N;
  P.n_coarse = im->nc; P.n_cells = im->ncell; P.n_surfaces = im->ns; P.N = im->N;
  h->coarse_fits_smem = sizeof(CoarseDev) * (size_t)im->nc <= 96 * 1024;   // 384 coarse faces; more are read through L1/L2 by the generic kernel
  h->face0 = im->face0;
  h->single_quad = im->nc == 1 && im->face0.kind == KIND_AFFINE_QUAD;
  h->queue_ok = h->coarse_fits_smem && im->n_affine + im->n_bilinear == im->nc;
  h->queue_general = im->n_bilinear > 0 || !im->nbr_complete;
  h->fast_ok = h->queue_ok && !h->queue_general;   // the FAST form of the general kernel: affine kinds with a complete neighbour table
  h->generic_ready = false;
  {
    // once per device and process: a few hundred cudaFuncSetAttribute calls cost milliseconds, and callers re-create the
    // handle for every trace
    ce = cudaSuccess;
    {
      std::lock_guard<std::mutex> lk(g_pool_mu);
      if (!g_kernels_configured[device_id & 63]) {
        ce = configure_trace_kernel(h->prop.sharedMemPerBlockOptin);
        g_kernels_configured[device_id & 63] = ce == cudaSuccess;
      }
    }
    if (ce != cudaSuccess) return bail(RTHX_ERR_CUDA, std::string("cudaFuncSetAttribute: ") + cudaGetErrorString(ce));   // bail re-takes the pool lock
  }
  if (im->needs_generic) {
    const int rc = ensure_generic(h);
    if (rc) return bail(rc, h->err);
  }
  if (sync && (ce = cudaStreamSynchronize(h->stream)) != cudaSuccess) return bail(RTHX_ERR_CUDA, std::string("mesh upload: ") + cudaGetErrorString(ce));
  *out = h;
  return RTHX_OK;
}

int check_mesh_args(const rthx_mesh* m) {
  if (!m || m->n_coarse < 1 || m->n_cells < 1 || m->n_bands < 1 || m->n_surfaces < 0 || !m->coarse_nv || !m->coarse_vx ||
      !m->coarse_vy || !m->coarse_solid || !m->fine_off || !m->cell_nv || !m->cell_vx || !m->cell_vy || !m->cell_mid ||
      !m->cell_volume || !m->cell_surf_id || !m->kappa || !m->sigma_s || !m->uniform_beta)
    return fail(nullptr, RTHX_ERR_ARG, "rthx_create: NULL or empty mesh field");
  return RTHX_OK;
}

}  // namespace

// Tables of the reference-faithful locator (uniform grids per fine-cell set, per-polygon normals): derived from the image on
// first use — at rthx_create for meshes with unverifiable lattices or more than 384 coarse faces, else by the first trace that
// asks for RTHX_LOCATOR_GENERIC or needs the generic kernel.  cfg3: 1.1 ms of host work that the analytic paths never pay.
// Host image of the generic tables, kept in a small most-recently-used cache keyed by a 128-bit hash of the geometry they are derived
// from (and of the grid knobs): callers re-create handles for every trace and rthx_create_multi makes one per device, but the tables
// of a mesh are built once per process (cfg3: ~25 ms of host work, 10 MB).
namespace {
struct GenericTables {
  std::vector<unsigned char> host;
  size_t o_sets = 0, o_bent = 0, o_bcand = 0, o_pnx = 0, o_pny = 0, o_frec = 0;
  uint64_t key[2] = {0, 0};
  int ncell = 0, nc = 0;
};
std::mutex g_gen_mu;
std::vector<std::shared_ptr<const GenericTables>> g_gen_cache;   // most recent first, at most 3 entries

void hash_bytes(uint64_t h[2], const void* data, size_t n) {    // two independent multiply-xorshift streams over 8-byte words
  const unsigned char* p = static_cast<const unsigned char*>(data);
  uint64_t a = h[0] ^ (n * 0x9E3779B97F4A7C15ull), b = h[1] + n;
  size_t i = 0;
  for (; i + 8 <= n; i += 8) {
    uint64_t w;
    std::memcpy(&w, p + i, 8);
    a = (a ^ w) * 0xFF51AFD7ED558CCDull; a ^= a >> 32;
    b = (b + w) * 0xC4CEB9FE1A85EC53ull; b ^= b >> 29;
  }
  uint64_t w = 0;
  if (i < n) std::memcpy(&w, p + i, n - i);
  a = (a ^ w) * 0xFF51AFD7ED558CCDull; a ^= a >> 33;
  b = (b + w) * 0xC4CEB9FE1A85EC53ull; b ^= b >> 31;
  h[0] = a; h[1] = b;
}

std::shared_ptr<const GenericTables> generic_tables(const HostImage& im) {
  const int nc = im.nc, ncell = im.ncell;
  const bool timing = std::getenv("RTHX_CREATE_TIMING") != nullptr;
  auto t_prev = std::chrono::steady_clock::now();
  auto lap = [&](const char* what) {
    if (!timing) return;
    const auto t = std::chrono::steady_clock::now();
    std::fprintf(stderr, "generic tables: %-24s %8.3f ms\n", what, std::chrono::duration<double, std::milli>(t - t_prev).count());
    t_prev = t;
  };
  uint64_t key[2] = {0x243F6A8885A308D3ull, 0x13198A2E03707344ull};
  hash_bytes(key, im.at<int32_t>(im.o_nv), 4 * (size_t)ncell);
  hash_bytes(key, im.at<double>(im.o_pvx), 32 * (size_t)ncell);
  hash_bytes(key, im.at<double>(im.o_pvy), 32 * (size_t)ncell);
  hash_bytes(key, im.at<double>(im.o_mid), 16 * (size_t)ncell);
  hash_bytes(key, im.at<double>(im.o_vol), 8 * (size_t)ncell);
  hash_bytes(key, im.at<int32_t>(im.o_surf), 16 * (size_t)ncell);
  hash_bytes(key, im.fine_off.data(), 4 * im.fine_off.size());
  for (const Poly& cp : im.coarse_polys) { const int32_t n = cp.n; hash_bytes(key, &n, 4); hash_bytes(key, cp.vx, 32); hash_bytes(key, cp.vy, 32); }   // (field by field: no padding bytes)
  for (const char* knob : {"RTHX_GRID_FINE", "RTHX_GRID_PER_FACE"}) { const char* ev = std::getenv(knob); hash_bytes(key, ev ? ev : "", ev ? std::strlen(ev) : 0); }
  {
    std::lock_guard<std::mutex> lk(g_gen_mu);
    for (size_t i = 0; i < g_gen_cache.size(); ++i) {
      const auto& t = g_gen_cache[i];
      if (t->key[0] == key[0] && t->key[1] == key[1] && t->ncell == ncell && t->nc == nc) {
        auto hit = t;
        g_gen_cache.erase(g_gen_cache.begin() + (long)i);
        g_gen_cache.insert(g_gen_cache.begin(), hit);
        return hit;
      }
    }
  }
  lap("hash + cache lookup");
  std::vector<Poly> polys((size_t)ncell + nc);
  const int32_t* nv = im.at<int32_t>(im.o_nv);
  const double* pvx = im.at<double>(im.o_pvx);
  const double* pvy = im.at<double>(im.o_pvy);
  const double* mid = im.at<double>(im.o_mid);
  const double* vol = im.at<double>(im.o_vol);
  for (int g = 0; g < ncell; ++g) {
    Poly& p = polys[g];
    p.n = nv[g];
    for (int i = 0; i < p.n; ++i) { p.vx[i] = pvx[4 * (size_t)g + i]; p.vy[i] = pvy[4 * (size_t)g + i]; }
    p.midx = mid[2 * (size_t)g]; p.midy = mid[2 * (size_t)g + 1]; p.volume = vol[g];
    poly_finish(p);
  }
  for (int c = 0; c < nc; ++c) polys[(size_t)ncell + c] = im.coarse_polys[c];
  lap("polygons + normals");
  std::vector<FaceSetDev> sets(1 + (size_t)nc);
  std::vector<int32_t> bent, bcand;
  build_grid(&polys[ncell], nc, ncell, sets[0], bent, bcand);
  for (int c = 0; c < nc; ++c) build_grid(&polys[im.fine_off[c]], im.fine_off[c + 1] - im.fine_off[c], im.fine_off[c], sets[1 + c], bent, bcand);
  lap("bucket grids");
  std::vector<double> pnx((size_t)ncell * 4), pny((size_t)ncell * 4), frec(polys.size() * FREC);
  const int32_t* surf = im.at<int32_t>(im.o_surf);
  for (size_t i = 0; i < polys.size(); ++i) {
    if (i < (size_t)ncell)
      for (int k = 0; k < 4; ++k) { pnx[4 * i + k] = polys[i].nx[k]; pny[4 * i + k] = polys[i].ny[k]; }
    face_record(polys[i], i < (size_t)ncell ? surf + 4 * i : nullptr, &frec[FREC * i]);
  }
  lap("polygon records");
  Arena A;
  A.host.reserve(sizeof(FaceSetDev) * sets.size() + 4 * (bent.size() + bcand.size()) + 8 * (pnx.size() + pny.size() + frec.size()) + 8 * 256);   // one allocation
  auto t = std::make_shared<GenericTables>();
  t->o_sets = A.add(sets); t->o_bent = A.add(bent); t->o_bcand = A.add(bcand); t->o_pnx = A.add(pnx); t->o_pny = A.add(pny); t->o_frec = A.add(frec);
  t->host = std::move(A.host);
  t->key[0] = key[0]; t->key[1] = key[1]; t->ncell = ncell; t->nc = nc;
  lap("table image");
  std::lock_guard<std::mutex> lk(g_gen_mu);
  g_gen_cache.insert(g_gen_cache.begin(), t);
  if (g_gen_cache.size() > 3) g_gen_cache.pop_back();
  return t;
}
}  // namespace

static void release_generic_cache() {
  std::lock_guard<std::mutex> lk(g_gen_mu);
  g_gen_cache.clear();
}

static int ensure_generic(rthx_handle* h) {
  if (h->generic_ready) return RTHX_OK;
  const HostImage& im = *h->image;
  const std::shared_ptr<const GenericTables> gt = generic_tables(im);
  struct { const std::vector<unsigned char>& host; size_t total; } A{gt->host, gt->host.size()};
  const size_t o_sets = gt->o_sets, o_bent = gt->o_bent, o_bcand = gt->o_bcand, o_pnx = gt->o_pnx, o_pny = gt->o_pny, o_frec = gt->o_frec;
  const bool timing = std::getenv("RTHX_CREATE_TIMING") != nullptr;
  const auto t_up = std::chrono::steady_clock::now();
  CU(h, cudaSetDevice(h->device));
  if (h->generic_cap < A.total) {
    cudaFree(h->generic_arena);
    h->generic_arena = nullptr; h->generic_cap = 0;
    CU(h, cudaMalloc(&h->generic_arena, A.total + A.total / 4));
    h->generic_cap = A.total + A.total / 4;
  }
  CU(h, cudaMemcpy(h->generic_arena, A.host.data(), A.host.size(), cudaMemcpyHostToDevice));
  if (timing) std::fprintf(stderr, "generic tables: %-24s %8.3f ms (%.1f MB)\n", "device arena + upload",
                           std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_up).count(), A.host.size() / 1e6);
  unsigned char* b8 = static_cast<unsigned char*>(h->generic_arena);
  TraceParams& P = h->base;
  P.sets = (const FaceSetDev*)(b8 + o_sets); P.bucket_ent = (const int4*)(b8 + o_bent); P.bucket_cand = (const int32_t*)(b8 + o_bcand);
  P.face_rec = (const double*)(b8 + o_frec);
  P.poly_nx = (const double*)(b8 + o_pnx); P.poly_ny = (const double*)(b8 + o_pny);
  h->mesh_bytes = im.bytes + A.host.size();
  h->generic_ready = true;
  return RTHX_OK;
}

extern "C" int rthx_device_count(int* n) {
  if (!n) return RTHX_ERR_ARG;
  *n = 0;
  int n_dev = 0;
  const cudaError_t ce = cudaGetDeviceCount(&n_dev);
  if (ce != cudaSuccess || n_dev == 0) { cudaGetLastError(); return fail(nullptr, RTHX_ERR_CUDA, std::string("no CUDA device (") + cudaGetErrorString(ce) + "); there is no CPU fallback"); }
  int usable = 0;
  for (int d = 0; d < n_dev; ++d) {
    int major = 0;
    if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, d) == cudaSuccess && major >= 10) ++usable;
  }
  *n = usable;
  return usable ? RTHX_OK : fail(nullptr, RTHX_ERR_CUDA, "no sm_100 class device (kernels are built for sm_100a only)");
}

extern "C" int rthx_create(rthx_handle** out, const rthx_mesh* m, int device_id) {
  if (!out) return fail(nullptr, RTHX_ERR_ARG, "rthx_create: out is NULL");
  *out = nullptr;
  return rthx_create_multi(out, m, &device_id, 1);
}

extern "C" int rthx_create_multi(rthx_handle** out, const rthx_mesh* m, const int* device_ids, int n) {
  if (!out || !device_ids || n < 1) return fail(nullptr, RTHX_ERR_ARG, "rthx_create_multi: bad argument");
  for (int i = 0; i < n; ++i) out[i] = nullptr;
  int rc = check_mesh_args(m);
  if (rc) return rc;
  int n_dev = 0;
  cudaError_t ce = cudaGetDeviceCount(&n_dev);
  if (ce != cudaSuccess || n_dev == 0)
    return fail(nullptr, RTHX_ERR_CUDA, std::string("rthx_create: no CUDA device (") + cudaGetErrorString(ce) + "); there is no CPU fallback");
  for (int i = 0; i < n; ++i) {
    if (device_ids[i] < 0 || device_ids[i] >= n_dev) return fail(nullptr, RTHX_ERR_ARG, "rthx_create: bad device id");
    for (int j = 0; j < i; ++j) if (device_ids[j] == device_ids[i]) return fail(nullptr, RTHX_ERR_ARG, "rthx_create_multi: duplicate device id");
  }
  int caller_device = 0;
  cudaGetDevice(&caller_device);
  struct RestoreDevice { int d; bool on; ~RestoreDevice() { if (on) cudaSetDevice(d); } } restore_device{caller_device, n > 1};   // a single-device create leaves that device current, as before
  const bool timing = std::getenv("RTHX_CREATE_TIMING") != nullptr;
  const auto t0 = std::chrono::steady_clock::now();
  std::shared_ptr<HostImage> im;
  std::string err;
  rc = prepare_mesh(m, im, err);
  if (rc) return fail(nullptr, rc, err);
  const auto t1 = std::chrono::steady_clock::now();
  auto undo = [&]() { for (int i = 0; i < n; ++i) { if (out[i]) rthx_destroy(out[i]); out[i] = nullptr; } };
  for (int i = 0; i < n; ++i) {
    rc = create_on_device(&out[i], im, device_ids[i], n_dev, /*sync=*/false);
    if (rc) { const std::string keep = g_create_err; undo(); g_create_err = keep; return rc; }
  }
  for (int i = 0; i < n; ++i) {       // every upload is in flight: wait for all of them
    cudaSetDevice(out[i]->device);
    if ((ce = cudaStreamSynchronize(out[i]->stream)) != cudaSuccess) { undo(); return fail(nullptr, RTHX_ERR_CUDA, std::string("mesh upload: ") + cudaGetErrorString(ce)); }
  }
  if (timing) {
    const auto t2 = std::chrono::steady_clock::now();
    std::fprintf(stderr, "rthx_create: host preparation %.3f ms, %d device(s) %.3f ms\n", std::chrono::duration<double, std::milli>(t1 - t0).count(), n,
                 std::chrono::duration<double, std::milli>(t2 - t1).count());
  }
  return RTHX_OK;
}

extern "C" int rthx_get_info(const rthx_handle* h, rthx_info* info) {
  if (!h || !info) return RTHX_ERR_ARG;
  info->n_elements = h->N; info->n_surfaces = h->ns; info->n_cells = h->n_cells; info->n_coarse = h->n_coarse;
  info->n_bands = h->n_bands; info->n_affine_faces = h->n_affine; info->device_id = h->device;
  info->sm_count = h->prop.multiProcessorCount; info->cc_major = h->prop.major; info->cc_minor = h->prop.minor;
  info->n_bilinear_faces = h->n_bilinear; info->reserved_ = 0;
  return RTHX_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// trace
// ---------------------------------------------------------------------------------------------------------------
namespace {

struct LaunchPlan { int n_owned, n_blocks, block_threads, row_chunks, hist_in_smem, fast, minb, multi, sq, queue_depth, queue_gen; size_t smem_bytes; };

int check_args(rthx_handle* h, const rthx_trace_args* a) {
  if (!a) return fail(h, RTHX_ERR_ARG, "trace: args is NULL");
  if (a->rays_per_emitter < 0) return fail(h, RTHX_ERR_ARG, "trace: rays_per_emitter out of range");
  if (a->n_bins < 1 || !a->bins) return fail(h, RTHX_ERR_ARG, "trace: n_bins must be >= 1");
  // the scratch regions behind the mesh image (bins, lost) are sized at rthx_create for 4 n_bands + 16 traced bins
  if ((size_t)a->n_bins > h->bins_cap || (size_t)a->n_bins * (size_t)h->N > h->lost_cap) return fail(h, RTHX_ERR_ARG, "trace: too many bins in one call (limit 4 * n_bands + 16)");
  for (int i = 0; i < a->n_bins; ++i) if (a->bins[i] < 0 || a->bins[i] >= h->n_bands) return fail(h, RTHX_ERR_ARG, "trace: band index out of range");
  if (a->mode != RTHX_FIRST_INTERACTION && a->mode != RTHX_MULTI_BOUNCE && a->mode != RTHX_MULTI_BOUNCE_SPECULAR) return fail(h, RTHX_ERR_ARG, "trace: unknown mode");
  if (a->mode != RTHX_FIRST_INTERACTION && !h->has_eps) return fail(h, RTHX_ERR_ARG, "trace: MULTI_BOUNCE needs rthx_mesh.epsilon");
  if (a->mode != RTHX_FIRST_INTERACTION && h->n_bands > 65535) return fail(h, RTHX_ERR_ARG, "trace: too many bands");
  if (a->emitter_world < 1 || a->emitter_rank < 0 || a->emitter_rank >= a->emitter_world) return fail(h, RTHX_ERR_ARG, "trace: bad emitter_rank/world");
  if (a->n_rec_ids < 0 || (a->n_rec_ids > 0 && !a->rec_ids)) return fail(h, RTHX_ERR_ARG, "trace: bad recorder ids");
  if (a->block_threads != 0 && (a->block_threads < 32 || a->block_threads > 256 || a->block_threads % 32)) return fail(h, RTHX_ERR_ARG, "trace: block_threads must be a multiple of 32 in [32,256]");
  if (a->row_chunks < 0) return fail(h, RTHX_ERR_ARG, "trace: row_chunks < 0");
  return RTHX_OK;
}

// where the resident counts come from
enum { RESIDENT_NONE = 0, RESIDENT_DENSE = 1, RESIDENT_SPARSE = 2, RESIDENT_HOST = 3, RESIDENT_MULTI = 4 };

void record_resident(rthx_handle* h, const rthx_trace_args* a, int kind) {
  h->resident_kind = kind;
  h->res_seed = a->seed; h->res_nudge = a->nudge; h->res_mode = a->mode; h->res_locator = a->locator;
  h->res_bins.assign(a->bins, a->bins + a->n_bins);
  h->ray_lo = a->ray_id_offset; h->ray_hi = a->ray_id_offset + a->rays_per_emitter;
}

// Preconditions of rthx_trace_exchange_continue: the resident counts are one trace of [ray_lo, ray_hi) that `a` continues
int check_continue(rthx_handle* h, const rthx_trace_args* a) {
  if (h->last_trace_bins <= 0 || h->resident_kind == RESIDENT_NONE)
    return fail(h, RTHX_ERR_ARG, "trace_continue: no resident counts (run rthx_trace_exchange with counts_out == NULL or rthx_trace_exchange_sparse first)");
  if (h->resident_kind == RESIDENT_HOST)
    return fail(h, RTHX_ERR_ARG, "trace_continue: the resident counts come from a host-output trace (counts_out != NULL); trace with counts_out == NULL to continue");
  if (h->resident_kind == RESIDENT_MULTI)
    return fail(h, RTHX_ERR_ARG, "trace_continue: the resident counts were gathered from several devices (rthx_trace_exchange_multi), whose peer hand-over stores rows instead of adding them");
  if (a->seed != h->res_seed) return fail(h, RTHX_ERR_ARG, "trace_continue: seed differs from the resident trace's");
  if (a->nudge != h->res_nudge) return fail(h, RTHX_ERR_ARG, "trace_continue: nudge differs from the resident trace's");
  if (a->mode != h->res_mode) return fail(h, RTHX_ERR_ARG, "trace_continue: mode differs from the resident trace's");
  if (a->locator != h->res_locator) return fail(h, RTHX_ERR_ARG, "trace_continue: locator differs from the resident trace's");
  if (a->n_bins != (int)h->res_bins.size() || !std::equal(a->bins, a->bins + a->n_bins, h->res_bins.begin()))
    return fail(h, RTHX_ERR_ARG, "trace_continue: bins differ from the resident trace's");
  if (a->emitter_rank != h->last_rank || a->emitter_world != h->last_world)
    return fail(h, RTHX_ERR_ARG, "trace_continue: emitter shard (emitter_rank / emitter_world) differs from the resident trace's");
  if (a->ray_id_offset != h->ray_hi)
    return fail(h, RTHX_ERR_ARG, "trace_continue: ray_id_offset " + std::to_string(a->ray_id_offset) + " does not continue the resident ray-id range [" +
                                     std::to_string(h->ray_lo) + ", " + std::to_string(h->ray_hi) + ")");
  if (a->rays_per_emitter > INT64_MAX - h->ray_hi) return fail(h, RTHX_ERR_ARG, "trace_continue: ray ids past 2^63");
  return RTHX_OK;
}

// variant bits of the queue kernel (rthx_kernels.cu, kernel_variant): 8 general faces, 16 generic locator (implies 8), 32 its 80-register build
int queue_variant_bits(const rthx_handle* h, const LaunchPlan& pl) {
  if (pl.queue_gen) return 8 + 16 + (pl.queue_gen == 3 ? 32 : 0);
  return h->queue_general ? 8 : 0;
}

// hash_slots > 0: the hashed row tally (no histogram, no SQ / queue kernels; the table takes hash_table_bytes(hash_slots))
LaunchPlan make_plan(const rthx_handle* h, const rthx_trace_args* a, int rank, int world, int hash_slots = 0) {
  LaunchPlan pl{};
  pl.n_owned = (h->N - rank + world - 1) / world;
  if (pl.n_owned < 0) pl.n_owned = 0;
  pl.block_threads = a->block_threads ? a->block_threads : 256;
  pl.fast = (h->fast_ok && a->locator != RTHX_LOCATOR_GENERIC) ? 1 : 0;
  pl.multi = a->mode != RTHX_FIRST_INTERACTION ? 1 : 0;
  pl.minb = pl.multi ? 2 : 4;
  if (const char* ev = std::getenv("RTHX_MINB")) { const int v = std::atoi(ev); if (v >= 2 && v <= 4) pl.minb = v; }   // tuning knob
  if (!pl.fast && !pl.multi) {     // generic locator kernel: 4 resident blocks (64 registers; +4 % with the sole-bucket locator) unless RTHX_GENERIC_MINB=3 (80 registers)
    pl.minb = 4;
    if (const char* ev = std::getenv("RTHX_GENERIC_MINB")) { if (std::atoi(ev) == 3) pl.minb = 3; }
  }
  const size_t coarse_bytes = h->coarse_fits_smem ? sizeof(CoarseDev) * (size_t)h->n_coarse : 0;
  const size_t hist_bytes = sizeof(uint32_t) * (size_t)h->N, em_bytes = sizeof(double) * 16 + 16 * (size_t)LOGTAB_N;   // emitter block + log table
  pl.hist_in_smem = (coarse_bytes + em_bytes + hist_bytes <= h->prop.sharedMemPerBlockOptin) ? 1 : 0;
  if (const char* ev = std::getenv("RTHX_FORCE_GLOBAL_TALLY")) { if (std::atoi(ev)) pl.hist_in_smem = 0; }   // test knob: the N > ~57k path
  if (hash_slots > 0) pl.hist_in_smem = 0;
  pl.sq = (h->single_quad && a->locator != RTHX_LOCATOR_GENERIC && pl.hist_in_smem) ? 1 : 0;
  if (const char* ev = std::getenv("RTHX_NO_SQ")) { if (std::atoi(ev)) pl.sq = 0; }   // test / tuning knob
  // MULTI_BOUNCE on any mesh with analytic locators runs in the queue kernel's MULTI variant (lanes refill when their ray is
  // absorbed); RTHX_MULTI_SQ=1 keeps the lock-step loop of the SQ kernel on single-quad domains (A/B knob)
  bool multi_queue = pl.multi && h->queue_ok && a->locator != RTHX_LOCATOR_GENERIC && pl.hist_in_smem && pl.block_threads == 256;
  if (const char* ev = std::getenv("RTHX_MULTI_SQ")) { if (std::atoi(ev) && pl.sq) multi_queue = false; }
  if (const char* ev = std::getenv("RTHX_QUEUE_DEPTH")) { if (std::atoi(ev) == 0 && !pl.sq) multi_queue = false; }
  if (multi_queue) pl.sq = 0;
  if (pl.sq && pl.multi) {
    pl.fast = 1; pl.minb = 4;                        // trace_exchange_sq_kernel<4, MULTI>
  } else if (pl.sq) {
    pl.fast = 1; pl.minb = 4;
    // tuning knob: 3 = the shared-loop SQ branch of the general kernel (A/B reference)
    if (const char* ev = std::getenv("RTHX_MINB")) { const int v = std::atoi(ev); if (v == 3) pl.minb = v; }
  }
  pl.smem_bytes = coarse_bytes + em_bytes + (pl.hist_in_smem ? hist_bytes : 0) + (hash_slots > 0 ? hash_table_bytes(hash_slots) : 0);
  // Multi-face FAST meshes: the queue kernel (per-warp ray queue in shared memory, 40 bytes per parked ray).  Depth = as many
  // rays per lane as still leave 4 resident blocks per SM, at most 8; RTHX_QUEUE_DEPTH overrides (0 = the lock-step kernel).
  // The same kernel's general variant also takes multi-face meshes through the GENERIC locator (faces without a verified lattice,
  // RTHX_LOCATOR_GENERIC) as long as the coarse descriptors fit in shared memory: a ray crosses several coarse faces there too, and
  // the lock-step kernel keeps 13 of 32 lanes busy.  RTHX_NO_QUEUE_GENERIC=1 keeps the lock-step kernel (A/B knob).
  pl.queue_gen = (!pl.multi && (a->locator == RTHX_LOCATOR_GENERIC || !h->queue_ok) && h->coarse_fits_smem && h->n_coarse > 1 &&
                  pl.hist_in_smem && pl.block_threads == 256) ? 1 : 0;
  if (const char* ev = std::getenv("RTHX_NO_QUEUE_GENERIC")) { if (std::atoi(ev)) pl.queue_gen = 0; }
  if (pl.queue_gen) { if (const char* ev = std::getenv("RTHX_GENERIC_MINB")) { if (std::atoi(ev) == 3) pl.queue_gen = 3; } }   // 3: the 80-register build (A/B knob)
  if (((h->queue_ok && a->locator != RTHX_LOCATOR_GENERIC && (!pl.multi || multi_queue) && (h->n_coarse > 1 || h->queue_general || multi_queue)) || pl.queue_gen) &&
      !pl.sq && pl.hist_in_smem && pl.block_threads == 256) {
    const size_t base = (pl.smem_bytes + 15) & ~size_t(15);
    const size_t per_depth = (size_t)pl.block_threads * (multi_queue ? 48 : 40);   // bytes per parked ray: p, d, S (+ ray index and event word for MULTI)
    // aim at 4 resident blocks per SM (3 for the MULTI variant, which is bounded to 85 registers); large descriptor tables /
    // histograms settle for fewer
    int depth = 0;
    const size_t max_depth = multi_queue ? 2 : 4;
    for (int blocks = multi_queue ? 3 : 4; blocks >= 1 && depth == 0; --blocks) {
      const size_t budget = std::min((size_t)h->prop.sharedMemPerMultiprocessor / blocks - 1024, (size_t)h->prop.sharedMemPerBlockOptin);
      if (base + per_depth <= budget) depth = (int)std::min<size_t>(max_depth, (budget - base) / per_depth);
    }
    if (const char* ev = std::getenv("RTHX_QUEUE_DEPTH")) { const int v = std::atoi(ev); if (v >= 0 && v <= (int)max_depth) depth = v; }
    if (depth == 3) depth = 2;                       // compiled depths: 1, 2, 4 rays per lane and batch (MULTI: 1, 2)
    if (depth >= (pl.queue_gen ? 2 : 1) && base + depth * per_depth <= h->prop.sharedMemPerBlockOptin) {   // (the generic variant is compiled for depths 2 and 4)
      pl.fast = 1; pl.minb = 6; pl.queue_depth = depth; pl.smem_bytes = base + depth * per_depth;
    }
  }
  if (!pl.queue_depth) pl.queue_gen = 0;
  const long long rows = (long long)pl.n_owned * a->n_bins;
  long long chunks = a->row_chunks;
  if (chunks <= 0) {
    // enough blocks for ~32 waves of the resident set, but keep >= 2048 rays (and >= N/2, the flush scan) per block
    const int per_sm = std::max(1, trace_kernel_max_blocks_per_sm(pl.block_threads, pl.smem_bytes, pl.hist_in_smem != 0, pl.fast != 0, pl.minb, pl.multi != 0, pl.sq != 0, pl.queue_depth + queue_variant_bits(h, pl),
                                                                  hash_slots > 0));
    const long long target = (long long)h->prop.multiProcessorCount * per_sm * 32;
    chunks = rows > 0 ? (target + rows - 1) / rows : 1;
    const long long min_rays = std::max<long long>(2048, h->N / 2);
    const long long max_chunks = std::max<long long>(1, a->rays_per_emitter / min_rays);
    chunks = std::max<long long>(1, std::min(chunks, max_chunks));
  }
  // A block's rays are counted in 32 bits (u32 row histogram, u32 loop counter advancing by blockDim.x): at most 2^31 rays per
  // block.  Auto-chosen chunk counts are raised to satisfy that; a plan that then exceeds the 1-D grid limit — or a caller-supplied
  // row_chunks that violates either bound — is rejected (n_blocks = -1 -> RTHX_ERR_ARG), never silently wrapped.
  if (a->row_chunks <= 0)
    while ((a->rays_per_emitter + chunks - 1) / chunks > 0x7FFFFFFFll) chunks *= 2;
  pl.row_chunks = (int)std::min<long long>(chunks, 0x7FFFFFFFll);
  if ((a->rays_per_emitter + chunks - 1) / chunks > 0x7FFFFFFFll || rows * chunks > 0x7FFFFFFFll) { pl.n_blocks = -1; return pl; }
  pl.n_blocks = (int)(rows * chunks);
  return pl;
}

void fill_params(const rthx_handle* h, const rthx_trace_args* a, const LaunchPlan& pl, int rank, int world, bool compact,
                 unsigned long long* counts, unsigned long long* lost, TraceParams& P) {
  P = h->base;
  P.bins = h->bins_dev;
  P.counts = counts; P.lost = lost;
  P.n_bins = a->n_bins;
  P.emitter_rank = rank; P.emitter_world = world; P.n_owned = pl.n_owned; P.y_offset = 0;
  P.compact_rows = compact ? 1 : 0;
  P.row_chunks = pl.row_chunks;
  P.queue_depth = pl.queue_depth;
  P.queue_bilinear = queue_variant_bits(h, pl);
  P.queue_refill = 24;
  if (const char* ev = std::getenv("RTHX_QUEUE_REFILL")) { const int v = std::atoi(ev); if (v >= 0 && v <= 32) P.queue_refill = v; }   // tuning knob
  P.coarse_in_smem = h->coarse_fits_smem ? 1 : 0;
  P.hist_in_smem = pl.hist_in_smem;
  P.force_generic = a->locator == RTHX_LOCATOR_GENERIC ? 1 : 0;
  P.multi_bounce = pl.multi; P.specular = a->mode == RTHX_MULTI_BOUNCE_SPECULAR ? 1 : 0;
  // a count matrix that lives on another GPU (fused peer flush) is updated with system-scope reductions
  P.flush_system = 0;
  cudaPointerAttributes pa;
  if (counts && cudaPointerGetAttributes(&pa, counts) == cudaSuccess && pa.type == cudaMemoryTypeDevice && pa.device != h->device) P.flush_system = 1;
  else cudaGetLastError();
  if (const char* ev = std::getenv("RTHX_FLUSH_SYSTEM")) P.flush_system = std::atoi(ev) ? 1 : 0;
  P.rec_bin = a->rec_bin;
  P.rays_per_emitter = a->rays_per_emitter;
  P.ray_id_offset = a->ray_id_offset;
  P.seed = a->seed;
  P.nudge = a->nudge;
  P.rec_slot = nullptr; P.rec_pts = nullptr; P.rec_valid = nullptr;
  P.face0 = h->face0;
  P.k_u52 = 1.0 - 0x1p-53; P.k_u32 = 1.0 - 0x1p-33; P.k_eps = 1e-10;
  P.k_u52c = 1.5 - 0x1p-53; P.k_u32c = 1.5 - 0x1p-33;
  {
    // SQ kernels: slab form of distToSurface2D on the single parallelogram — centre line and half width of each edge pair
    // (h0 - q = hw - (q - cen), q - h2 = hw + (q - cen)), the folded lattice-inverse offsets, and the axis-aligned special case
    // (n0 = (0, +-1), n1 = (+-1, 0), lattice axes along x and y, all exact: every product with a zero component vanishes exactly,
    // so the shortened arithmetic is bit-identical to the general form).
    const CoarseDev& f = h->face0;
    P.sq_cen0 = 0.5 * (f.h[0] + f.h[2]); P.sq_hw0 = 0.5 * (f.h[0] - f.h[2]);
    P.sq_cen1 = 0.5 * (f.h[1] + f.h[3]); P.sq_hw1 = 0.5 * (f.h[1] - f.h[3]);
    P.sq_lc1 = -(f.ax * f.g1x + f.ay * f.g1y);
    P.sq_lc2 = -(f.ax * f.g2x + f.ay * f.g2y);
    P.sq_one_m_nudge = 1.0 - a->nudge;
    const bool axis = f.nx[0] == 0.0 && std::fabs(f.ny[0]) == 1.0 && std::fabs(f.nx[1]) == 1.0 && f.ny[1] == 0.0 && f.g1y == 0.0 && f.g2x == 0.0;
    P.sq_axis = axis ? 1 : 0;
    if (const char* ev = std::getenv("RTHX_NO_AXIS")) { if (std::atoi(ev)) P.sq_axis = 0; }   // test knob: the general SQ loop
    P.queue_sq = (h->single_quad && pl.multi && pl.queue_depth > 0) ? (P.sq_axis ? 1 : 2) : 0;
    if (const char* ev = std::getenv("RTHX_NO_QUEUE_SQ")) { if (std::atoi(ev)) P.queue_sq = 0; }   // A/B knob: the generic step on a single quad
    P.sq_cy = f.ny[0] * P.sq_cen0; P.sq_cx = f.nx[1] * P.sq_cen1;
    P.sq_flip0 = f.ny[0] < 0.0 ? 0x80000000u : 0u; P.sq_flip1 = f.nx[1] < 0.0 ? 0x80000000u : 0u;
  }
  uint32_t k0 = (uint32_t)a->seed, k1 = (uint32_t)(a->seed >> 32);
  for (int r = 0; r < 10; ++r) { P.rk[2 * r] = k0; P.rk[2 * r + 1] = k1; k0 += 0x9E3779B9u; k1 += 0xBB67AE85u; }
}

template <class T>
cudaError_t ensure(T** ptr, size_t* cap, size_t need) {
  if (*cap >= need && *ptr) return cudaSuccess;
  if (*ptr) cudaFree(*ptr);
  *ptr = nullptr; *cap = 0;
  cudaError_t e = cudaMalloc((void**)ptr, std::max<size_t>(need, 1) * sizeof(T));
  if (e == cudaSuccess) *cap = need;
  return e;
}

void fill_stats(rthx_stats* st, const LaunchPlan& pl, const rthx_trace_args* a) {
  if (!st) return;
  std::memset(st, 0, sizeof(*st));
  st->rays_traced = (int64_t)pl.n_owned * a->n_bins * a->rays_per_emitter;
  st->n_blocks = pl.n_blocks; st->block_threads = pl.block_threads; st->row_chunks = pl.row_chunks;
  st->smem_bytes = (int32_t)pl.smem_bytes; st->hist_in_smem = pl.hist_in_smem;
}

// Enqueue (zero +) kernel for one handle on `stream`; counts layout compact (owned rows) or full.
// [y0, y1) restricts the launch to a range of owned-emitter ordinals (y1 < 0: all rows).
int enqueue_trace(rthx_handle* h, const rthx_trace_args* a, int rank, int world, bool compact, unsigned long long* counts,
                  unsigned long long* lost, int zero_first, bool with_rec, int n_rec_slots, cudaStream_t stream,
                  LaunchPlan* plan_out, int* n_launches, int y0 = 0, int y1 = -1, bool upload_bins = true) {
  LaunchPlan pl = make_plan(h, a, rank, world);
  if (pl.n_blocks < 0) return fail(h, RTHX_ERR_ARG, "trace: rays_per_emitter / row_chunks out of range (a block traces at most 2^31 rays, a launch at most 2^31 blocks)");
  if (!pl.fast || pl.queue_gen) { const int rcg = ensure_generic(h); if (rcg) return rcg; }     // the generic kernel reads the reference-faithful locator tables
  if (upload_bins) CU(h, cudaMemcpyAsync(h->bins_dev, a->bins, sizeof(int32_t) * (size_t)a->n_bins, cudaMemcpyHostToDevice, stream));
  // A matrix in peer memory (fused multi-GPU flush) is never the target of reductions: the chunks of a row add up in a local
  // compact staging matrix and the finished row is handed over with plain stores (flush_row_hist) — so the peer rows need no
  // clearing either.  Without the shared-memory histogram (N > ~57 k) the old path stays: system-scope atomics into zeroed rows.
  // (a CUDA-IPC mapping reports the mapping device, not the owner: such callers say so with RTHX_DEST_PEER)
  bool peer = (zero_first & RTHX_DEST_PEER) != 0;
  zero_first &= ~RTHX_DEST_PEER;
  {
    cudaPointerAttributes pa;
    if (counts && cudaPointerGetAttributes(&pa, counts) == cudaSuccess && pa.type == cudaMemoryTypeDevice && pa.device != h->device) peer = true;
    else cudaGetLastError();
    if (const char* ev = std::getenv("RTHX_FLUSH_SYSTEM")) peer = std::atoi(ev) != 0;     // test knob: exercise the hand-over on one GPU
    if (const char* ev = std::getenv("RTHX_PEER_ATOMICS")) { if (std::atoi(ev)) peer = false; }   // A/B knob: the old red.sys flush
  }
  const bool staged = peer && pl.hist_in_smem && !compact;
  unsigned long long* stage_counts = nullptr;
  unsigned int* row_done = nullptr;
  if (staged) {
    h->last_trace_bins = 0; h->csr_bin = -1; h->csc_bin = -1; h->sparse_counts = false;   // counts_dev becomes the staging matrix
    const size_t n_rows = (size_t)a->n_bins * (size_t)pl.n_owned;
    if (pl.row_chunks > 1) {
      CU(h, ensure(&h->counts_dev, &h->counts_cap, n_rows * (size_t)h->N));
      CU(h, cudaMemsetAsync(h->counts_dev, 0, sizeof(unsigned long long) * n_rows * (size_t)h->N, stream));
      stage_counts = h->counts_dev;
      *n_launches += 1;
    }
    CU(h, ensure(&h->row_done_dev, &h->row_done_cap, std::max<size_t>(n_rows, 1)));
    CU(h, cudaMemsetAsync(h->row_done_dev, 0, sizeof(unsigned int) * std::max<size_t>(n_rows, 1), stream));
    row_done = h->row_done_dev;
  }
  const size_t rows = compact ? (size_t)pl.n_owned : (size_t)h->N;
  if (zero_first == RTHX_ZERO_ALL) {
    CU(h, cudaMemsetAsync(counts, 0, sizeof(unsigned long long) * (size_t)a->n_bins * rows * h->N, stream));
    CU(h, cudaMemsetAsync(lost, 0, sizeof(unsigned long long) * (size_t)a->n_bins * h->N, stream));
    *n_launches += 2;
  } else if (zero_first == RTHX_ZERO_OWN_ROWS && pl.n_owned > 0) {
    // rows e = rank + y*world: a strided 2-D memset per traced bin (works on peer-mapped memory too)
    const size_t rb = sizeof(unsigned long long) * (size_t)h->N;
    for (int b = 0; b < a->n_bins; ++b) {
      if (compact) {
        CU(h, cudaMemsetAsync(counts + (size_t)b * pl.n_owned * h->N, 0, rb * pl.n_owned, stream));
      } else if (!staged) {
        CU(h, cudaMemset2DAsync(counts + ((size_t)b * h->N + rank) * h->N, rb * world, 0, rb, (size_t)pl.n_owned, stream));
      }
      CU(h, cudaMemset2DAsync(lost + (size_t)b * h->N + rank, sizeof(unsigned long long) * world, 0, sizeof(unsigned long long), (size_t)pl.n_owned, stream));
      *n_launches += 2;
    }
  }
  TraceParams P;
  fill_params(h, a, pl, rank, world, compact, counts, lost, P);
  if (staged) {
    P.peer_counts = counts; P.row_done = row_done;
    P.counts = stage_counts; P.compact_rows = 1;                         // nullptr with row_chunks == 1: rows are written out directly
    P.flush_system = 1;                                                  // the lost counters live next to the peer matrix
  }
  if (with_rec && n_rec_slots > 0) { P.rec_slot = h->rec_slot_dev; P.rec_pts = h->rec_pts_dev; P.rec_valid = h->rec_valid_dev; }
  if (y1 < 0) y1 = pl.n_owned;
  P.y_offset = y0;
  const long long nb = (long long)(y1 - y0) * a->n_bins * pl.row_chunks;
  CU(h, launch_trace_exchange(P, (int)nb, pl.block_threads, pl.smem_bytes, pl.fast != 0, pl.minb, pl.sq != 0, stream));
  if (nb > 0) *n_launches += 1;
  *plan_out = pl;
  return RTHX_OK;
}

// Host-output trace of one handle, pipelined (pipeline_launch + pipeline_copy): the owned rows are cut into batches whose kernels alternate between two
// compute streams (so the tail of one batch overlaps the head of the next) and whose device->host copies run on a third
// stream as soon as the batch's kernel has finished.  All work is enqueued; the caller synchronises copy_stream.
//   ev[0] start, ev[1] first kernel start, ev[2] last kernel end, ev[3] last copy end.
// Row range of batch b of the pipelined host-output trace.  The last four batches are a quarter of the others: what follows the
// last kernel is the device->host copy of the last batch only, so a short last batch shortens the tail of the call (cfg3: 56 MB
// -> 17 MB behind the last kernel).  Fewer than 8 batches are split evenly.
void batch_rows_of(int n_owned, int n_batches, int b, int& y0, int& y1) {
  if (n_batches < 8) {
    y0 = (int)((long long)n_owned * b / n_batches); y1 = (int)((long long)n_owned * (b + 1) / n_batches);
    return;
  }
  const long long units = 4LL * (n_batches - 4) + 4;            // full batches weigh 4, the last four 1
  auto edge = [&](int k) { return k <= n_batches - 4 ? 4LL * k : 4LL * (n_batches - 4) + (k - (n_batches - 4)); };
  y0 = (int)((long long)n_owned * edge(b) / units); y1 = (int)((long long)n_owned * edge(b + 1) / units);
}

int pipeline_launch(rthx_handle* h, const rthx_trace_args* a, int rank, int world, bool with_rec, int n_slots,
                    LaunchPlan* plan_out, int* n_launches, int* n_batches_out) {
  const int N = h->N;
  const int n_owned = (N - rank + world - 1) / world;
  // counts_dev is about to be overwritten: whatever view an earlier trace left behind (resident bins, CSR row pointers) is void
  // until the caller re-validates it (rthx_trace_exchange does, for a complete single-device trace)
  h->last_trace_bins = 0; h->csr_bin = -1; h->csc_bin = -1; h->sparse_counts = false;
  CU(h, ensure(&h->counts_dev, &h->counts_cap, (size_t)a->n_bins * (size_t)n_owned * N));
  LaunchPlan pl = make_plan(h, a, rank, world);
  if (pl.n_blocks < 0) return fail(h, RTHX_ERR_ARG, "trace: rays_per_emitter / row_chunks out of range (a block traces at most 2^31 rays, a launch at most 2^31 blocks)");
  // batches: >= ~2 waves of resident blocks each, at most 16 (consecutive batches alternate between two streams, so a batch's
  // draining tail overlaps the next one's head; cfg3 at 1e10 rays: 16 batches, the copy behind the last kernel is 17 MB and the
  // call ends 0.5 ms after the kernel — with 5 even batches it was 180 MB and 3.6 ms)
  const int per_sm = std::max(1, trace_kernel_max_blocks_per_sm(pl.block_threads, pl.smem_bytes, pl.hist_in_smem != 0, pl.fast != 0, pl.minb, pl.multi != 0, pl.sq != 0, pl.queue_depth + queue_variant_bits(h, pl)));
  const long long resident = (long long)h->prop.multiProcessorCount * per_sm;
  int n_batches = (int)std::min<long long>(16, std::max<long long>(1, pl.n_blocks / (2 * resident)));
  n_batches = std::max(1, std::min(n_batches, n_owned));
  if (const char* ev = std::getenv("RTHX_BATCHES")) { const int v = std::atoi(ev); if (v >= 1 && v <= 16) n_batches = std::min(v, std::max(1, n_owned)); }
  CU(h, cudaMemcpyAsync(h->bins_dev, a->bins, sizeof(int32_t) * (size_t)a->n_bins, cudaMemcpyHostToDevice, h->stream));
  CU(h, cudaMemsetAsync(h->counts_dev, 0, sizeof(unsigned long long) * (size_t)a->n_bins * (size_t)n_owned * N, h->stream));
  CU(h, cudaMemsetAsync(h->lost_dev, 0, sizeof(unsigned long long) * (size_t)a->n_bins * N, h->stream));
  *n_launches += 2;
  CU(h, cudaEventRecord(h->ev[1], h->stream));
  CU(h, cudaStreamWaitEvent(h->stream2, h->ev[1], 0));
  for (int b = 0; b < n_batches; ++b) {
    int y0, y1;
    batch_rows_of(n_owned, n_batches, b, y0, y1);
    cudaStream_t cs = (b & 1) ? h->stream2 : h->stream;
    LaunchPlan tmp{};
    int rc = enqueue_trace(h, a, rank, world, /*compact=*/true, h->counts_dev, h->lost_dev, RTHX_ZERO_NONE, with_rec, n_slots, cs, &tmp, n_launches, y0, y1,
                           /*upload_bins=*/false);
    if (rc) return rc;
    CU(h, cudaEventRecord(h->bev[b], cs));
  }
  // last kernel end = both compute streams drained
  CU(h, cudaEventRecord(h->bev[16], h->stream2));
  CU(h, cudaStreamWaitEvent(h->stream, h->bev[16], 0));
  CU(h, cudaEventRecord(h->ev[2], h->stream));
  *plan_out = pl;
  *n_batches_out = n_batches;
  return RTHX_OK;
}

void parallel_memcpy(void* dst, const void* src, size_t bytes) {
  const int nt = bytes >= (size_t(16) << 20) ? 4 : 1;
  if (nt == 1) { std::memcpy(dst, src, bytes); return; }
  std::vector<std::thread> th;
  const size_t per = ((bytes / nt) + 4095) & ~size_t(4095);
  for (int t = 0; t < nt; ++t) {
    const size_t off = (size_t)t * per;
    if (off >= bytes) break;
    const size_t n = std::min(per, bytes - off);
    th.emplace_back([=] { std::memcpy((char*)dst + off, (const char*)src + off, n); });
  }
  for (auto& t : th) t.join();
}

// Second half of the pipeline: copy each batch's rows to the caller's matrix as soon as its kernel has finished.
//   pinned / registered destination : cudaMemcpy(2D)Async straight into it on copy_stream (nothing blocks the host);
//   pageable destination (e.g. a Julia Array): DMA into two pinned staging buffers, the host thread moves batch b-1 to
//       the caller's memory while batch b is in flight (a pageable cudaMemcpyAsync would block the host per batch and
//       crawl at ~4 GB/s).
int pipeline_copy(rthx_handle* h, const rthx_trace_args* a, int rank, int world, uint64_t* counts_out, int n_batches) {
  const int N = h->N;
  const int n_owned = (N - rank + world - 1) / world;
  cudaPointerAttributes pa;
  bool pinned = cudaPointerGetAttributes(&pa, counts_out) == cudaSuccess && (pa.type == cudaMemoryTypeHost || pa.type == cudaMemoryTypeManaged);
  cudaGetLastError();
  if (const char* ev = std::getenv("RTHX_FORCE_STAGING")) { if (std::atoi(ev)) pinned = false; }
  const size_t row_bytes = sizeof(uint64_t) * (size_t)N;
  auto batch_rows = [&](int b, int& y0, int& y1) { batch_rows_of(n_owned, n_batches, b, y0, y1); };
  if (pinned) {
    for (int b = 0; b < n_batches; ++b) {
      int y0, y1; batch_rows(b, y0, y1);
      CU(h, cudaStreamWaitEvent(h->copy_stream, h->bev[b], 0));
      for (int bin = 0; bin < a->n_bins && y1 > y0; ++bin) {
        const unsigned long long* src = h->counts_dev + ((size_t)bin * n_owned + y0) * N;
        if (world == 1)
          CU(h, cudaMemcpyAsync(counts_out + ((size_t)bin * N + y0) * N, src, row_bytes * (size_t)(y1 - y0), cudaMemcpyDeviceToHost, h->copy_stream));
        else
          CU(h, cudaMemcpy2DAsync(counts_out + ((size_t)bin * N + rank + (size_t)y0 * world) * N, row_bytes * world, src, row_bytes, row_bytes,
                                  (size_t)(y1 - y0), cudaMemcpyDeviceToHost, h->copy_stream));
      }
    }
    CU(h, cudaStreamWaitEvent(h->copy_stream, h->ev[2], 0));
    return RTHX_OK;
  }
  // staged path
  size_t max_rows = 0;
  for (int b = 0; b < n_batches; ++b) { int y0, y1; batch_rows(b, y0, y1); max_rows = std::max(max_rows, (size_t)(y1 - y0)); }
  const size_t stage_bytes = std::max<size_t>(1, max_rows * a->n_bins * row_bytes);
  if (h->stage_cap < stage_bytes) {
    for (auto& sp : h->stage) { if (sp) cudaFreeHost(sp); sp = nullptr; }
    h->stage_cap = 0;
    for (auto& sp : h->stage) CU(h, cudaMallocHost(&sp, stage_bytes));
    h->stage_cap = stage_bytes;
  }
  auto unload = [&](int b) {   // staging[b&1] -> caller's matrix
    int y0, y1; batch_rows(b, y0, y1);
    const size_t rows = (size_t)(y1 - y0);
    const char* st = (const char*)h->stage[b & 1];
    for (int bin = 0; bin < a->n_bins && rows; ++bin) {
      const char* src = st + (size_t)bin * rows * row_bytes;
      if (world == 1) parallel_memcpy(counts_out + ((size_t)bin * N + y0) * N, src, rows * row_bytes);
      else
        for (size_t r = 0; r < rows; ++r) std::memcpy(counts_out + ((size_t)bin * N + rank + (size_t)(y0 + r) * world) * N, src + r * row_bytes, row_bytes);
    }
  };
  for (int b = 0; b < n_batches; ++b) {
    int y0, y1; batch_rows(b, y0, y1);
    const size_t rows = (size_t)(y1 - y0);
    CU(h, cudaStreamWaitEvent(h->copy_stream, h->bev[b], 0));
    for (int bin = 0; bin < a->n_bins && rows; ++bin)
      CU(h, cudaMemcpyAsync((char*)h->stage[b & 1] + (size_t)bin * rows * row_bytes, h->counts_dev + ((size_t)bin * n_owned + y0) * N, rows * row_bytes,
                            cudaMemcpyDeviceToHost, h->copy_stream));
    CU(h, cudaEventRecord(h->cev[b & 1], h->copy_stream));
    if (b >= 1) { CU(h, cudaEventSynchronize(h->cev[(b - 1) & 1])); unload(b - 1); }
  }
  CU(h, cudaEventSynchronize(h->cev[(n_batches - 1) & 1]));
  unload(n_batches - 1);
  CU(h, cudaStreamWaitEvent(h->copy_stream, h->ev[2], 0));
  return RTHX_OK;
}

// Recorder slots: rank (0..n_rec-1) of each recorded element in ascending element order, -1 elsewhere.
int prepare_recorder(rthx_handle* h, const rthx_trace_args* a, rthx_rec_out* rec, int* n_slots, cudaStream_t stream) {
  *n_slots = 0;
  if (!rec || a->n_rec_ids <= 0) return RTHX_OK;
  std::vector<int32_t> slot(h->N, -1);
  for (int i = 0; i < a->n_rec_ids; ++i) if (a->rec_ids[i] >= 0 && a->rec_ids[i] < h->N) slot[a->rec_ids[i]] = 0;
  int n = 0;
  for (int e = 0; e < h->N; ++e) if (slot[e] == 0) slot[e] = n++;
  *n_slots = n;
  if (n == 0) return RTHX_OK;
  const size_t pts = (size_t)n * (size_t)a->rays_per_emitter;
  CU(h, ensure(&h->rec_pts_dev, &h->rec_pts_cap, pts * 4));
  CU(h, ensure(&h->rec_valid_dev, &h->rec_valid_cap, pts));
  CU(h, cudaMemcpyAsync(h->rec_slot_dev, slot.data(), sizeof(int32_t) * (size_t)h->N, cudaMemcpyHostToDevice, stream));
  CU(h, cudaMemsetAsync(h->rec_valid_dev, 0, pts, stream));
  return RTHX_OK;
}

int collect_recorder(rthx_handle* h, const rthx_trace_args* a, rthx_rec_out* rec, int n_slots, cudaStream_t stream, bool append) {
  if (!rec) return RTHX_OK;
  if (!append) rec->n_recorded = 0;
  if (n_slots == 0) return RTHX_OK;
  const size_t pts = (size_t)n_slots * (size_t)a->rays_per_emitter;
  std::vector<double> buf(pts * 4);
  std::vector<uint8_t> valid(pts);
  CU(h, cudaMemcpyAsync(buf.data(), h->rec_pts_dev, sizeof(double) * pts * 4, cudaMemcpyDeviceToHost, stream));
  CU(h, cudaMemcpyAsync(valid.data(), h->rec_valid_dev, pts, cudaMemcpyDeviceToHost, stream));
  CU(h, cudaStreamSynchronize(stream));
  for (size_t s = 0; s < pts; ++s) {
    if (!valid[s]) continue;
    if (rec->n_recorded >= rec->capacity) break;
    const int64_t k = rec->n_recorded++;
    rec->origins[2 * k] = buf[4 * s]; rec->origins[2 * k + 1] = buf[4 * s + 1];
    rec->endpoints[2 * k] = buf[4 * s + 2]; rec->endpoints[2 * k + 1] = buf[4 * s + 3];
  }
  return RTHX_OK;
}

}  // namespace

extern "C" int rthx_trace_exchange(rthx_handle* h, const rthx_trace_args* a, uint64_t* counts_out, uint64_t* lost_out,
                                   rthx_rec_out* rec, rthx_stats* st) {
  if (!h) return RTHX_ERR_ARG;
  int rc = check_args(h, a);
  if (rc) return rc;
  CU(h, cudaSetDevice(h->device));
  const int N = h->N;
  int n_slots = 0, n_launches = 0;
  CU(h, cudaEventRecord(h->ev[0], h->stream));
  rc = prepare_recorder(h, a, rec, &n_slots, h->stream);
  if (rc) return rc;
  LaunchPlan pl{};
  int n_batches = 1;
  rc = pipeline_launch(h, a, a->emitter_rank, a->emitter_world, rec != nullptr, n_slots, &pl, &n_launches, &n_batches);
  if (rc) return rc;
  if (counts_out) {
    rc = pipeline_copy(h, a, a->emitter_rank, a->emitter_world, counts_out, n_batches);
    if (rc) return rc;
  } else {
    CU(h, cudaStreamWaitEvent(h->copy_stream, h->ev[2], 0));
  }
  // the (compact) rows this call owns stay resident: all of them for a plain trace, those of a shard / row tile otherwise
  h->last_trace_bins = a->n_bins;
  h->last_trace_rows = (size_t)pl.n_owned; h->last_rank = a->emitter_rank; h->last_world = a->emitter_world;
  h->csr_bin = -1; h->csc_bin = -1;
  record_resident(h, a, counts_out ? RESIDENT_HOST : RESIDENT_DENSE);
  std::vector<uint64_t> lost_host((size_t)a->n_bins * N);
  CU(h, cudaMemcpyAsync(lost_host.data(), h->lost_dev, sizeof(uint64_t) * lost_host.size(), cudaMemcpyDeviceToHost, h->copy_stream));
  CU(h, cudaEventRecord(h->ev[3], h->copy_stream));
  CU(h, cudaStreamSynchronize(h->copy_stream));
  CU(h, cudaStreamSynchronize(h->stream));
  if (lost_out) std::memcpy(lost_out, lost_host.data(), sizeof(uint64_t) * lost_host.size());
  rc = collect_recorder(h, a, rec, n_slots, h->stream, false);
  if (rc) return rc;
  if (st) {
    fill_stats(st, pl, a);
    float ms = 0;
    CU(h, cudaEventElapsedTime(&ms, h->ev[1], h->ev[2])); st->kernel_ms = ms;
    CU(h, cudaEventElapsedTime(&ms, h->ev[0], h->ev[3])); st->total_ms = ms;
    int64_t nl = 0;
    for (uint64_t v : lost_host) nl += (int64_t)v;
    st->rays_lost = nl;
    st->n_launches = n_launches;
  }
  return RTHX_OK;
}

extern "C" int rthx_trace_exchange_device(rthx_handle* h, const rthx_trace_args* a, void* counts_dev, void* lost_dev, void* stream,
                                          int zero_first, rthx_stats* st) {
  if (!h) return RTHX_ERR_ARG;
  int rc = check_args(h, a);
  if (rc) return rc;
  if (!counts_dev || !lost_dev) return fail(h, RTHX_ERR_ARG, "trace_device: NULL device buffer");
  CU(h, cudaSetDevice(h->device));
  LaunchPlan pl{};
  int n_launches = 0;
  rc = enqueue_trace(h, a, a->emitter_rank, a->emitter_world, /*compact=*/false, (unsigned long long*)counts_dev,
                     (unsigned long long*)lost_dev, zero_first, false, 0, (cudaStream_t)stream, &pl, &n_launches);
  if (rc) return rc;
  if (st) { fill_stats(st, pl, a); st->n_launches = n_launches; }
  return RTHX_OK;
}

namespace {
// grow a device array to >= need elements, keeping its first `keep`
template <class T>
cudaError_t grow_keep(T** ptr, size_t* cap, size_t need, size_t keep, cudaStream_t st) {
  if (*cap >= need && *ptr) return cudaSuccess;
  size_t nc = std::max(need, *cap + *cap / 2);
  T* np = nullptr;
  if (cudaMalloc((void**)&np, std::max<size_t>(nc, 1) * sizeof(T)) != cudaSuccess) {
    cudaGetLastError();
    nc = need;
    cudaError_t e = cudaMalloc((void**)&np, std::max<size_t>(nc, 1) * sizeof(T));
    if (e != cudaSuccess) return e;
  }
  cudaError_t e = cudaSuccess;
  if (keep && *ptr) e = cudaMemcpyAsync(np, *ptr, keep * sizeof(T), cudaMemcpyDeviceToDevice, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) { cudaFree(np); return e; }
  cudaFree(*ptr);
  *ptr = np; *cap = nc;
  return cudaSuccess;
}
}  // namespace

namespace {
// What one hashed-tally pass over the rows of a call did (sparse_trace_rows)
struct SparseRun {
  LaunchPlan pl{};
  int log2s = 0, groups = 0, n_slots = 0, n_launches = 0;
  long long cap = 0, n_rows = 0, total = 0, pairs = 0, flushes = 0;
  double kernel_ms = 0, reduce_ms = 0;
};

// A device array freed when it goes out of scope (scratch of rthx_trace_exchange_continue)
template <class T>
struct DevBuf {
  T* p = nullptr;
  size_t cap = 0;
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  ~DevBuf() { cudaFree(p); }
};

// Trace the rows of `a` with the hashed row tally and append the sorted unique (key, u64 total) pairs of every row group to
// (*out_keys, *out_vals), growing them as needed; lost_dev is cleared first and counts the rays of this call.  A group whose pairs
// overran the pair buffer is traced again split in two.  ev[0] marks the start of the call's device work.
int sparse_trace_rows(rthx_handle* h, const rthx_trace_args* a, rthx_rec_out* rec, unsigned long long** out_keys, size_t* keys_cap,
                      unsigned long long** out_vals, size_t* vals_cap, SparseRun& R) {
  const int N = h->N, nb = a->n_bins, rank = a->emitter_rank, world = a->emitter_world;
  const int bt = a->block_threads ? a->block_threads : 256;
  int log2s = 12;                                            // 4096 slots: 32 KB of table
  int min_log2s = 1;
  while ((1 << min_log2s) < 2 * bt) ++min_log2s;             // a round of blockDim.x inserts must fit below half full
  bool forced = false;
  if (const char* ev = std::getenv("RTHX_SPARSE_HASH_SLOTS")) {   // test knob: small tables flush many times
    const long long v = std::atoll(ev);
    if (v > 0) { log2s = 0; while ((1ll << log2s) < v) ++log2s; forced = true; }
  }
  log2s = std::max(log2s, min_log2s);
  LaunchPlan pl = make_plan(h, a, rank, world, 1 << log2s);
  if (pl.n_blocks < 0) return fail(h, RTHX_ERR_ARG, "trace: rays_per_emitter / row_chunks out of range (a block traces at most 2^31 rays, a launch at most 2^31 blocks)");
  if (!forced) {                                             // a block with few rays needs no large table: clearing and scanning it is the cost
    const long long per_block = (a->rays_per_emitter + pl.row_chunks - 1) / pl.row_chunks;
    const long long distinct = std::min<long long>(per_block, N);
    const int old = log2s;
    while (log2s > min_log2s && (1ll << (log2s - 1)) >= 2 * distinct) --log2s;
    pl.smem_bytes = pl.smem_bytes - hash_table_bytes(1 << old) + hash_table_bytes(1 << log2s);
  }
  if (pl.smem_bytes > h->prop.sharedMemPerBlockOptin) return fail(h, RTHX_ERR_ARG, "trace_sparse: hash table does not fit in shared memory");
  if (!pl.fast) { const int rcg = ensure_generic(h); if (rcg) return rcg; }
  // pair buffer: at most one pair per tallied ray, and at most half the free device memory (24 bytes a pair with the sort's
  // alternate buffers); the other half is left for the resident totals
  long long cap = 0x7FFFFFFFll;
  {
    size_t free_b = 0, total_b = 0;
    CU(h, cudaMemGetInfo(&free_b, &total_b));
    const double rays = (double)pl.n_owned * nb * (double)a->rays_per_emitter;
    cap = (long long)std::min<double>((double)cap, std::min(rays, (double)(free_b / 2 + h->sk_pairs_cap * 24) / 24.0));
    if (const char* ev = std::getenv("RTHX_SPARSE_PAIR_CAP")) { const long long v = std::atoll(ev); if (v > 0) cap = std::min(cap, v); }   // test knob: forces row-group splits
    cap = std::max<long long>(cap, 1);
  }
  if ((size_t)cap > h->sk_pairs_cap) {
    cudaFree(h->sk_pairs); h->sk_pairs = nullptr; h->sk_pairs_cap = 0;
    CU(h, cudaMalloc(&h->sk_pairs, (size_t)cap * 24));
    h->sk_pairs_cap = (size_t)cap;
  }
  CU(h, ensure(&h->sk_ctl, &h->sk_ctl_cap, 4));
  const size_t tmp_bytes = tally_temp_bytes(cap);
  CU(h, ensure(reinterpret_cast<char**>(&h->sk_tmp), &h->sk_tmp_cap, tmp_bytes));
  unsigned long long* keys = (unsigned long long*)h->sk_pairs;
  unsigned long long* keys_alt = keys + cap;
  uint32_t* cnt = (uint32_t*)(keys_alt + cap);
  uint32_t* cnt_alt = cnt + cap;
  const long long n_rows = (long long)pl.n_owned * nb;       // row key y * n_bins + bi
  int end_bit = 32;
  while ((1ll << (end_bit - 32)) < n_rows) ++end_bit;

  CU(h, cudaEventRecord(h->ev[0], h->stream));
  int rc = prepare_recorder(h, a, rec, &R.n_slots, h->stream);
  if (rc) return rc;
  CU(h, cudaMemcpyAsync(h->bins_dev, a->bins, sizeof(int32_t) * (size_t)nb, cudaMemcpyHostToDevice, h->stream));
  CU(h, cudaMemsetAsync(h->lost_dev, 0, sizeof(unsigned long long) * (size_t)nb * N, h->stream));
  R.n_launches += 1;
  TraceParams P;
  fill_params(h, a, pl, rank, world, true, nullptr, h->lost_dev, P);
  if (R.n_slots > 0) { P.rec_slot = h->rec_slot_dev; P.rec_pts = h->rec_pts_dev; P.rec_valid = h->rec_valid_dev; }
  P.sk_keys = keys; P.sk_cnt = cnt; P.sk_ctl = h->sk_ctl; P.sk_cap = (unsigned long long)cap; P.sk_slots_log2 = log2s;

  // row groups in ascending order: a group whose pairs overran the buffer is traced again as two halves
  std::vector<std::pair<int, int>> todo{{0, pl.n_owned}};
  long long total = 0;
  while (!todo.empty()) {
    const auto [y0, y1] = todo.front();
    todo.erase(todo.begin());
    if (y1 <= y0) continue;
    CU(h, cudaMemsetAsync(h->sk_ctl, 0, 4 * sizeof(unsigned long long), h->stream));
    P.y_offset = y0;
    CU(h, cudaEventRecord(h->ev[1], h->stream));
    CU(h, launch_trace_exchange(P, (int)((long long)(y1 - y0) * nb * pl.row_chunks), pl.block_threads, pl.smem_bytes, pl.fast != 0, pl.minb, false, h->stream));
    CU(h, cudaEventRecord(h->ev[2], h->stream));
    R.n_launches += 2;
    unsigned long long ctl[4];
    CU(h, cudaMemcpyAsync(ctl, h->sk_ctl, sizeof(ctl), cudaMemcpyDeviceToHost, h->stream));
    CU(h, cudaStreamSynchronize(h->stream));
    float ms = 0;
    CU(h, cudaEventElapsedTime(&ms, h->ev[1], h->ev[2])); R.kernel_ms += ms;
    if (ctl[1]) {
      if (y1 - y0 == 1) return fail(h, RTHX_ERR_NOMEM, "trace_sparse: the pairs of one emitter row exceed the pair buffer (" + std::to_string(cap) + " pairs)");
      for (int b = 0; b < nb; ++b)                          // the lost rays of the group are counted again
        CU(h, cudaMemset2DAsync(h->lost_dev + (size_t)b * N + rank + (size_t)y0 * world, sizeof(unsigned long long) * world, 0,
                                sizeof(unsigned long long), (size_t)(y1 - y0), h->stream));
      const int mid = y0 + (y1 - y0) / 2;
      todo.insert(todo.begin(), {{y0, mid}, {mid, y1}});
      continue;
    }
    const long long n = (long long)ctl[0];
    ++R.groups; R.pairs += n; R.flushes += (long long)ctl[2];
    CU(h, grow_keep(out_keys, keys_cap, (size_t)(total + std::max(n, 1ll)), (size_t)total, h->stream));
    CU(h, grow_keep(out_vals, vals_cap, (size_t)(total + std::max(n, 1ll)), (size_t)total, h->stream));
    CU(h, cudaEventRecord(h->ev[1], h->stream));
    CU(h, tally_reduce(keys, cnt, keys_alt, cnt_alt, n, end_bit, *out_keys + total, *out_vals + total, (long long*)(h->sk_ctl + 3), h->sk_tmp,
                       h->sk_tmp_cap, h->stream));
    CU(h, cudaEventRecord(h->ev[2], h->stream));
    long long uniq = 0;
    CU(h, cudaMemcpyAsync(&uniq, h->sk_ctl + 3, sizeof(long long), cudaMemcpyDeviceToHost, h->stream));
    CU(h, cudaStreamSynchronize(h->stream));
    CU(h, cudaEventElapsedTime(&ms, h->ev[1], h->ev[2])); R.reduce_ms += ms;
    total += uniq;
  }
  R.pl = pl; R.log2s = log2s; R.cap = cap; R.n_rows = n_rows; R.total = total;
  return RTHX_OK;
}

// Second half of a hashed-tally trace or continuation whose sorted unique pairs (R.total of them) are in sk_keys / sk_vals: row
// pointers, lost read-out, handle state, recorder and statistics.  lost_before (continuation): the lost counts of the resident
// trace, added to this call's.
int sparse_finish(rthx_handle* h, const rthx_trace_args* a, const SparseRun& R, const std::vector<uint64_t>* lost_before, uint64_t* lost_out,
                  rthx_rec_out* rec, rthx_stats* st, rthx_sparse_stats* sst) {
  const int N = h->N, nb = a->n_bins;
  CU(h, ensure(&h->sk_rowptr, &h->sk_rowptr_cap, (size_t)R.n_rows + 1));
  CU(h, tally_row_ptr(h->sk_keys, R.total, R.n_rows, h->sk_rowptr, h->stream));
  std::vector<uint64_t> lost_host((size_t)nb * N);
  CU(h, cudaMemcpyAsync(lost_host.data(), h->lost_dev, sizeof(uint64_t) * lost_host.size(), cudaMemcpyDeviceToHost, h->stream));
  if (lost_before) {
    CU(h, cudaStreamSynchronize(h->stream));
    for (size_t k = 0; k < lost_host.size(); ++k) lost_host[k] += (*lost_before)[k];
    CU(h, cudaMemcpyAsync(h->lost_dev, lost_host.data(), sizeof(uint64_t) * lost_host.size(), cudaMemcpyHostToDevice, h->stream));
  }
  CU(h, cudaEventRecord(h->ev[3], h->stream));
  CU(h, cudaStreamSynchronize(h->stream));
  h->sparse_counts = true; h->sk_nnz = R.total;
  h->last_trace_bins = nb; h->last_trace_rows = (size_t)R.pl.n_owned; h->last_rank = a->emitter_rank; h->last_world = a->emitter_world;
  if (lost_before) h->ray_hi += a->rays_per_emitter;
  else record_resident(h, a, RESIDENT_SPARSE);
  if (lost_out) std::memcpy(lost_out, lost_host.data(), sizeof(uint64_t) * lost_host.size());
  int rc = collect_recorder(h, a, rec, R.n_slots, h->stream, false);
  if (rc) return rc;
  if (st) {
    fill_stats(st, R.pl, a);
    st->kernel_ms = R.kernel_ms;
    float ms = 0;
    CU(h, cudaEventElapsedTime(&ms, h->ev[0], h->ev[3])); st->total_ms = ms;
    int64_t nl = 0;
    for (uint64_t v : lost_host) nl += (int64_t)v;
    st->rays_lost = nl;
    st->n_launches = R.n_launches;
  }
  if (sst) {
    std::memset(sst, 0, sizeof(*sst));
    sst->pairs = R.pairs; sst->nnz = R.total; sst->flushes = R.flushes; sst->pair_capacity = R.cap;
    sst->row_groups = R.groups; sst->hash_slots = 1 << R.log2s; sst->reduce_ms = R.reduce_ms;
  }
  return RTHX_OK;
}

// Continuation of a hashed-tally trace, up to the merged set: the new rays' pairs are reduced into a set of their own, which is then
// merged into the resident set (equal keys summed) and replaces it as the last step.  R.total receives the merged key count.
int continue_sparse_merge(rthx_handle* h, const rthx_trace_args* a, rthx_rec_out* rec, long long old_nnz, SparseRun& R) {
  DevBuf<unsigned long long> add_keys, add_vals;
  int rc = sparse_trace_rows(h, a, rec, &add_keys.p, &add_keys.cap, &add_vals.p, &add_vals.cap, R);
  if (rc) return rc;
  // the merge does not use the pair buffer: when device memory is short it makes room for the merged set
  auto alloc = [h](void** p, size_t bytes) {
    cudaError_t e = cudaMalloc(p, bytes);
    if (e == cudaErrorMemoryAllocation && h->sk_pairs) {
      cudaGetLastError();
      cudaFree(h->sk_pairs); h->sk_pairs = nullptr; h->sk_pairs_cap = 0;
      e = cudaMalloc(p, bytes);
    }
    return e;
  };
  const long long n_out = old_nnz + R.total, n_tiles = tally_merge_tiles(n_out);
  DevBuf<unsigned long long> mrg_keys, mrg_vals;
  DevBuf<long long> tiles;
  CU(h, alloc((void**)&mrg_keys.p, sizeof(unsigned long long) * (size_t)std::max(n_out, 1ll)));
  CU(h, alloc((void**)&mrg_vals.p, sizeof(unsigned long long) * (size_t)std::max(n_out, 1ll)));
  CU(h, alloc((void**)&tiles.p, sizeof(long long) * 2 * (size_t)(n_tiles + 1)));
  mrg_keys.cap = mrg_vals.cap = (size_t)std::max(n_out, 1ll);
  CU(h, ensure(reinterpret_cast<char**>(&h->sk_tmp), &h->sk_tmp_cap, tally_merge_temp_bytes(n_tiles)));
  CU(h, cudaEventRecord(h->ev[1], h->stream));
  CU(h, tally_merge(h->sk_keys, h->sk_vals, old_nnz, add_keys.p, add_vals.p, R.total, mrg_keys.p, mrg_vals.p, tiles.p, h->sk_tmp, h->sk_tmp_cap,
                    h->stream));
  CU(h, cudaEventRecord(h->ev[2], h->stream));
  long long merged = 0;
  CU(h, cudaMemcpyAsync(&merged, tiles.p + 2 * n_tiles + 1, sizeof(long long), cudaMemcpyDeviceToHost, h->stream));
  CU(h, cudaStreamSynchronize(h->stream));
  float ms = 0;
  CU(h, cudaEventElapsedTime(&ms, h->ev[1], h->ev[2]));
  R.reduce_ms += ms;
  R.n_launches += n_tiles > 0 ? 5 : 3;     // memset, scan (init + scan kernel), and the counting and writing passes
  R.total = merged;
  std::swap(h->sk_keys, mrg_keys.p); std::swap(h->sk_keys_cap, mrg_keys.cap);   // the old set is freed with mrg_*
  std::swap(h->sk_vals, mrg_vals.p); std::swap(h->sk_vals_cap, mrg_vals.cap);
  return RTHX_OK;
}

// Continuation of a hashed-tally trace.  Until the merged set replaces it the resident set is untouched, so a failure before that
// point leaves it resident, with its lost counters restored.
int continue_sparse(rthx_handle* h, const rthx_trace_args* a, uint64_t* lost_out, rthx_rec_out* rec, rthx_stats* st, rthx_sparse_stats* sst) {
  std::vector<uint64_t> lost_before((size_t)a->n_bins * h->N);
  CU(h, cudaMemcpyAsync(lost_before.data(), h->lost_dev, sizeof(uint64_t) * lost_before.size(), cudaMemcpyDeviceToHost, h->stream));
  CU(h, cudaStreamSynchronize(h->stream));
  const long long old_nnz = h->sk_nnz;
  const int old_bins = h->last_trace_bins;
  h->last_trace_bins = 0; h->csr_bin = -1; h->csc_bin = -1;  // incomplete until the merge has landed
  SparseRun R;
  const int rc = continue_sparse_merge(h, a, rec, old_nnz, R);
  if (rc) {
    if (cudaMemcpy(h->lost_dev, lost_before.data(), sizeof(uint64_t) * lost_before.size(), cudaMemcpyHostToDevice) == cudaSuccess)
      h->last_trace_bins = old_bins;
    else
      cudaGetLastError();
    return rc;
  }
  return sparse_finish(h, a, R, &lost_before, lost_out, rec, st, sst);
}

// Continuation of a dense resident trace: the same launches as rthx_trace_exchange(counts_out == NULL) without clearing the counts or
// the lost counters.  Every flush into a matrix on the handle's own device adds (shared-memory histogram rows, global atomics,
// row_chunks == 1 alike), so the counts add up to those of one trace of the whole range.
int continue_dense(rthx_handle* h, const rthx_trace_args* a, uint64_t* lost_out, rthx_rec_out* rec, rthx_stats* st) {
  int n_slots = 0, n_launches = 0;
  CU(h, cudaEventRecord(h->ev[0], h->stream));
  int rc = prepare_recorder(h, a, rec, &n_slots, h->stream);
  if (rc) return rc;
  h->last_trace_bins = 0; h->csr_bin = -1; h->csc_bin = -1;  // incomplete until the kernels have finished
  CU(h, cudaEventRecord(h->ev[1], h->stream));
  LaunchPlan pl{};
  rc = enqueue_trace(h, a, a->emitter_rank, a->emitter_world, /*compact=*/true, h->counts_dev, h->lost_dev, RTHX_ZERO_NONE, rec != nullptr, n_slots,
                     h->stream, &pl, &n_launches);
  if (rc) return rc;
  CU(h, cudaEventRecord(h->ev[2], h->stream));
  std::vector<uint64_t> lost_host((size_t)a->n_bins * h->N);
  CU(h, cudaMemcpyAsync(lost_host.data(), h->lost_dev, sizeof(uint64_t) * lost_host.size(), cudaMemcpyDeviceToHost, h->stream));
  CU(h, cudaEventRecord(h->ev[3], h->stream));
  CU(h, cudaStreamSynchronize(h->stream));
  h->last_trace_bins = a->n_bins;
  h->ray_hi += a->rays_per_emitter;
  if (lost_out) std::memcpy(lost_out, lost_host.data(), sizeof(uint64_t) * lost_host.size());
  rc = collect_recorder(h, a, rec, n_slots, h->stream, false);
  if (rc) return rc;
  if (st) {
    fill_stats(st, pl, a);
    float ms = 0;
    CU(h, cudaEventElapsedTime(&ms, h->ev[1], h->ev[2])); st->kernel_ms = ms;
    CU(h, cudaEventElapsedTime(&ms, h->ev[0], h->ev[3])); st->total_ms = ms;
    int64_t nl = 0;
    for (uint64_t v : lost_host) nl += (int64_t)v;
    st->rays_lost = nl;
    st->n_launches = n_launches;
  }
  return RTHX_OK;
}
}  // namespace

extern "C" int rthx_trace_exchange_sparse(rthx_handle* h, const rthx_trace_args* a, uint64_t* lost_out, rthx_rec_out* rec, rthx_stats* st,
                                          rthx_sparse_stats* sst) {
  if (!h) return RTHX_ERR_ARG;
  int rc = check_args(h, a);
  if (rc) return rc;
  if (a->mode != RTHX_FIRST_INTERACTION)
    return fail(h, RTHX_ERR_ARG, "trace_sparse: the hashed tally supports RTHX_FIRST_INTERACTION only (trace MULTI_BOUNCE with rthx_trace_exchange)");
  CU(h, cudaSetDevice(h->device));
  // whatever counts were resident (dense or sparse) are void from here on
  h->last_trace_bins = 0; h->csr_bin = -1; h->csc_bin = -1; h->sparse_counts = false; h->sk_nnz = 0;
  SparseRun R;
  rc = sparse_trace_rows(h, a, rec, &h->sk_keys, &h->sk_keys_cap, &h->sk_vals, &h->sk_vals_cap, R);
  if (rc) return rc;
  return sparse_finish(h, a, R, nullptr, lost_out, rec, st, sst);
}

extern "C" int rthx_trace_exchange_continue(rthx_handle* h, const rthx_trace_args* a, uint64_t* lost_out, rthx_rec_out* rec, rthx_stats* st,
                                            rthx_sparse_stats* sst) {
  if (!h) return RTHX_ERR_ARG;
  int rc = check_args(h, a);
  if (rc) return rc;
  rc = check_continue(h, a);
  if (rc) return rc;
  CU(h, cudaSetDevice(h->device));
  if (h->sparse_counts) return continue_sparse(h, a, lost_out, rec, st, sst);
  if (sst) std::memset(sst, 0, sizeof(*sst));
  return continue_dense(h, a, lost_out, rec, st);
}

namespace {

// Per-device outcome of rthx_trace_exchange_multi (one host thread drives each device).
struct MultiJob {
  int rc = RTHX_OK;
  std::string err;
  LaunchPlan plan{};
  int slots = 0, batches = 1, launches = 0;
  double kernel_ms = 0, total_ms = 0;
  std::vector<uint64_t> lost;
};

// Recorder read-back of one device in a multi-device trace: every device holds slots for all recorded elements, only the rows it
// owns were written.  Appends one chunk per owned recorded element.
struct RecChunk { int elem; std::vector<double> o, e; };

int gather_recorder(rthx_handle* h, const rthx_trace_args* a, int rank, int world, int n_slots, std::vector<RecChunk>& chunks) {
  if (n_slots <= 0) return RTHX_OK;
  const int N = h->N;
  const size_t rpe = (size_t)a->rays_per_emitter, pts = (size_t)n_slots * rpe;
  std::vector<double> buf(pts * 4);
  std::vector<uint8_t> valid(pts);
  CU(h, cudaMemcpy(buf.data(), h->rec_pts_dev, sizeof(double) * pts * 4, cudaMemcpyDeviceToHost));
  CU(h, cudaMemcpy(valid.data(), h->rec_valid_dev, pts, cudaMemcpyDeviceToHost));
  std::vector<int32_t> slot(N, -1);
  for (int k = 0; k < a->n_rec_ids; ++k) if (a->rec_ids[k] >= 0 && a->rec_ids[k] < N) slot[a->rec_ids[k]] = 0;
  int ord = 0;
  for (int e = 0; e < N; ++e) {
    if (slot[e] != 0) continue;
    const int s_ = ord++;
    if (e % world != rank) continue;
    RecChunk c; c.elem = e;
    for (size_t r = 0; r < rpe; ++r) {
      const size_t s = (size_t)s_ * rpe + r;
      if (!valid[s]) continue;
      c.o.push_back(buf[4 * s]); c.o.push_back(buf[4 * s + 1]); c.e.push_back(buf[4 * s + 2]); c.e.push_back(buf[4 * s + 3]);
    }
    chunks.push_back(std::move(c));
  }
  return RTHX_OK;
}

}  // namespace

// Single-process multi-GPU trace.  One host thread per device enqueues that device's work and drains its copies, so neither the
// launch sequences (a few dozen driver calls each) nor the staging of a pageable destination serialise across devices.
//   counts_out != NULL : every device traces its rows e = i (mod n) into a compact matrix of its own and copies exactly those rows
//                        into the caller's matrix (pipelined behind the kernels, each over its own PCIe link).  The rows tile the
//                        matrix, so nothing is cleared on the host and nothing is reduced.
//   counts_out == NULL : the devices flush their rows straight into ONE matrix in the memory of hs[0]'s device through peer access
//                        (NVLink / NVSwitch, system-scope red.add.u64 fused into the trace kernel).  The complete matrix stays
//                        resident on hs[0] for rthx_counts_csr / rthx_counts_csc / rthx_smooth_* / rthx_solve_grey.
extern "C" int rthx_trace_exchange_multi(rthx_handle** hs, int n, const rthx_trace_args* a, uint64_t* counts_out, uint64_t* lost_out,
                                         rthx_rec_out* rec, rthx_stats* st) {
  if (!hs || n < 1 || !hs[0]) return RTHX_ERR_ARG;
  rthx_handle* h0 = hs[0];
  int rc = check_args(h0, a);
  if (rc) return rc;
  const int N = h0->N;
  for (int i = 0; i < n; ++i) {
    if (!hs[i] || hs[i]->N != N || hs[i]->n_bands != h0->n_bands) return fail(h0, RTHX_ERR_ARG, "trace_multi: handles differ");
    for (int j = 0; j < i; ++j) if (hs[j] == hs[i]) return fail(h0, RTHX_ERR_ARG, "trace_multi: the same handle twice");   // several handles on one device are fine
  }
  int caller_device = 0;
  cudaGetDevice(&caller_device);
  struct RestoreDevice { int d; ~RestoreDevice() { cudaSetDevice(d); } } restore_device{caller_device};   // whatever path returns
  const bool gather = counts_out == nullptr;
  const size_t lost_n = (size_t)a->n_bins * N;
  std::vector<MultiJob> jobs(n);
  unsigned long long* shared_counts = nullptr;
  if (gather) {
    // the full matrix lives on hs[0]; the other devices need peer access to it
    CU(h0, cudaSetDevice(h0->device));
    h0->last_trace_bins = 0; h0->csr_bin = -1; h0->csc_bin = -1; h0->sparse_counts = false;
    CU(h0, ensure(&h0->counts_dev, &h0->counts_cap, (size_t)a->n_bins * (size_t)N * N));
    shared_counts = h0->counts_dev;
    for (int i = 1; i < n; ++i) {
      hs[i]->last_trace_bins = 0; hs[i]->csr_bin = -1; hs[i]->csc_bin = -1; hs[i]->sparse_counts = false;
      if (hs[i]->device == h0->device) continue;
      int can = 0;
      CU(h0, cudaDeviceCanAccessPeer(&can, hs[i]->device, h0->device));
      if (!can) return fail(h0, RTHX_ERR_CUDA, "trace_multi: no peer access between the devices (pass a host matrix instead)");
      CU(h0, cudaSetDevice(hs[i]->device));
      const cudaError_t pe = cudaDeviceEnablePeerAccess(h0->device, 0);
      if (pe != cudaSuccess && pe != cudaErrorPeerAccessAlreadyEnabled) return fail(h0, RTHX_ERR_CUDA, std::string("cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(pe));
      cudaGetLastError();
    }
    // nothing is cleared centrally: every device clears its own rows / lost counters (device 0 in place, the others need no
    // clearing of the matrix at all — they hand finished rows over with plain stores)
  }
  auto device_job = [&](int i) {
    rthx_handle* h = hs[i];
    MultiJob& J = jobs[i];
    auto run = [&]() -> int {
      CU(h, cudaSetDevice(h->device));
      CU(h, cudaEventRecord(h->ev[0], h->stream));
      int r = prepare_recorder(h, a, rec, &J.slots, h->stream);
      if (r) return r;
      if (gather) {
        CU(h, cudaEventRecord(h->ev[1], h->stream));
        r = enqueue_trace(h, a, i, n, /*compact=*/false, shared_counts, h0->lost_dev, RTHX_ZERO_OWN_ROWS, rec != nullptr, J.slots, h->stream, &J.plan, &J.launches);
        if (r) return r;
        CU(h, cudaEventRecord(h->ev[2], h->stream));
        CU(h, cudaEventRecord(h->ev[3], h->stream));
        CU(h, cudaStreamSynchronize(h->stream));
      } else {
        r = pipeline_launch(h, a, i, n, rec != nullptr, J.slots, &J.plan, &J.launches, &J.batches);
        if (r) return r;
        r = pipeline_copy(h, a, i, n, counts_out, J.batches);
        if (r) return r;
        J.lost.resize(lost_n);
        CU(h, cudaMemcpyAsync(J.lost.data(), h->lost_dev, sizeof(uint64_t) * lost_n, cudaMemcpyDeviceToHost, h->copy_stream));
        CU(h, cudaEventRecord(h->ev[3], h->copy_stream));
        CU(h, cudaStreamSynchronize(h->copy_stream));
        CU(h, cudaStreamSynchronize(h->stream));
      }
      float ms = 0;
      CU(h, cudaEventElapsedTime(&ms, h->ev[1], h->ev[2])); J.kernel_ms = ms;
      CU(h, cudaEventElapsedTime(&ms, h->ev[0], h->ev[3])); J.total_ms = ms;
      return RTHX_OK;
    };
    J.rc = run();
    if (J.rc) J.err = h->err;
  };
  {
    // one host thread per device; if the process cannot start threads the devices are driven in turn (slower, still correct) —
    // no C++ exception may cross the C ABI
    std::vector<std::thread> th;
    std::vector<int> inline_jobs;
    for (int i = 1; i < n; ++i) {
      try { th.emplace_back(device_job, i); } catch (...) { inline_jobs.push_back(i); }
    }
    device_job(0);
    for (int i : inline_jobs) device_job(i);
    for (auto& t : th) t.join();
  }
  for (int i = 0; i < n; ++i) if (jobs[i].rc) return fail(h0, jobs[i].rc, jobs[i].err);
  std::vector<uint64_t> lost_sum(lost_n, 0);
  if (gather) {
    CU(h0, cudaSetDevice(h0->device));
    CU(h0, cudaMemcpy(lost_sum.data(), h0->lost_dev, sizeof(uint64_t) * lost_n, cudaMemcpyDeviceToHost));
    h0->last_trace_bins = a->n_bins; h0->last_trace_rows = (size_t)N; h0->last_rank = 0; h0->last_world = 1;
    record_resident(h0, a, RESIDENT_MULTI);
  } else {
    for (int i = 0; i < n; ++i)
      for (size_t k = 0; k < lost_n; ++k) lost_sum[k] += jobs[i].lost[k];
  }
  if (rec) {
    // recorded rays must come out in ascending element order: gather per device, then merge by element
    rec->n_recorded = 0;
    std::vector<RecChunk> chunks;
    for (int i = 0; i < n; ++i) {
      CU(h0, cudaSetDevice(hs[i]->device));
      rc = gather_recorder(hs[i], a, i, n, jobs[i].slots, chunks);
      if (rc) return fail(h0, rc, hs[i]->err);
    }
    std::sort(chunks.begin(), chunks.end(), [](const RecChunk& x, const RecChunk& y) { return x.elem < y.elem; });
    for (auto& c : chunks)
      for (size_t k = 0; k < c.o.size(); k += 2) {
        if (rec->n_recorded >= rec->capacity) break;
        const int64_t q = rec->n_recorded++;
        rec->origins[2 * q] = c.o[k]; rec->origins[2 * q + 1] = c.o[k + 1];
        rec->endpoints[2 * q] = c.e[k]; rec->endpoints[2 * q + 1] = c.e[k + 1];
      }
  }
  if (lost_out) std::memcpy(lost_out, lost_sum.data(), sizeof(uint64_t) * lost_n);
  if (st) {
    fill_stats(st, jobs[0].plan, a);
    st->rays_traced = (int64_t)N * a->n_bins * a->rays_per_emitter;
    int64_t nl = 0;
    for (uint64_t v : lost_sum) nl += (int64_t)v;
    st->rays_lost = nl;
    int nbk = 0, nlaunch = 0;
    double kmax = 0, tmax = 0;
    for (auto& J : jobs) { nbk += J.plan.n_blocks; nlaunch += J.launches; kmax = std::max(kmax, J.kernel_ms); tmax = std::max(tmax, J.total_ms); }
    st->n_blocks = nbk; st->n_launches = nlaunch;
    st->kernel_ms = kmax; st->total_ms = tmax;     // the slowest device
  }
  return RTHX_OK;
}

extern "C" int rthx_set_copy_helpers(rthx_handle* h, rthx_handle** helpers, int n) {
  if (!h || n < 0 || (n > 0 && !helpers)) return RTHX_ERR_ARG;
  h->helpers.clear();
  for (int i = 0; i < n; ++i) {
    if (!helpers[i] || helpers[i] == h) return fail(h, RTHX_ERR_ARG, "set_copy_helpers: bad helper handle");
    if (helpers[i]->device != h->device) h->helpers.push_back(helpers[i]);     // a helper on the same device has no link of its own
  }
  return RTHX_OK;
}

extern "C" int rthx_host_alloc(void** ptr, uint64_t bytes) {
  if (!ptr || bytes == 0) return fail(nullptr, RTHX_ERR_ARG, "rthx_host_alloc: bad argument");
  *ptr = nullptr;
  cudaError_t e = cudaHostAlloc(ptr, (size_t)bytes, cudaHostAllocPortable);
  if (e != cudaSuccess) { cudaGetLastError(); return fail(nullptr, e == cudaErrorMemoryAllocation ? RTHX_ERR_NOMEM : RTHX_ERR_CUDA, std::string("cudaHostAlloc: ") + cudaGetErrorString(e)); }
  return RTHX_OK;
}

extern "C" int rthx_host_free(void* ptr) {
  if (!ptr) return RTHX_OK;
  cudaError_t e = cudaFreeHost(ptr);
  if (e != cudaSuccess) return fail(nullptr, RTHX_ERR_CUDA, std::string("cudaFreeHost: ") + cudaGetErrorString(e));
  return RTHX_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// peer-memory plumbing (CUDA IPC) for the fused flush
// ---------------------------------------------------------------------------------------------------------------
#define CUG(call)                                                                                     \
  do {                                                                                                \
    cudaError_t e_ = (call);                                                                          \
    if (e_ != cudaSuccess) return fail(nullptr, RTHX_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); \
  } while (0)

extern "C" int rthx_host_register(void* ptr, uint64_t bytes) {
  if (!ptr || bytes == 0) return fail(nullptr, RTHX_ERR_ARG, "rthx_host_register: bad argument");
  CUG(cudaHostRegister(ptr, (size_t)bytes, cudaHostRegisterPortable));
  return RTHX_OK;
}

extern "C" int rthx_host_unregister(void* ptr) {
  if (!ptr) return RTHX_OK;
  CUG(cudaHostUnregister(ptr));
  return RTHX_OK;
}

extern "C" int rthx_shared_alloc(int device_id, uint64_t bytes, void** dev_ptr, unsigned char ipc_handle[64]) {
  if (!dev_ptr || !ipc_handle || bytes == 0) return fail(nullptr, RTHX_ERR_ARG, "rthx_shared_alloc: bad argument");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "CUDA IPC handle is 64 bytes");
  CUG(cudaSetDevice(device_id));
  void* p = nullptr;
  CUG(cudaMalloc(&p, (size_t)bytes));
  cudaIpcMemHandle_t hnd;
  cudaError_t e = cudaIpcGetMemHandle(&hnd, p);
  if (e != cudaSuccess) { cudaFree(p); return fail(nullptr, RTHX_ERR_CUDA, std::string("cudaIpcGetMemHandle: ") + cudaGetErrorString(e)); }
  std::memcpy(ipc_handle, &hnd, 64);
  *dev_ptr = p;
  return RTHX_OK;
}

extern "C" int rthx_shared_open(int device_id, const unsigned char ipc_handle[64], void** dev_ptr) {
  if (!dev_ptr || !ipc_handle) return fail(nullptr, RTHX_ERR_ARG, "rthx_shared_open: bad argument");
  CUG(cudaSetDevice(device_id));
  cudaIpcMemHandle_t hnd;
  std::memcpy(&hnd, ipc_handle, 64);
  void* p = nullptr;
  CUG(cudaIpcOpenMemHandle(&p, hnd, cudaIpcMemLazyEnablePeerAccess));
  *dev_ptr = p;
  return RTHX_OK;
}

extern "C" int rthx_shared_close(int device_id, void* dev_ptr) {
  if (!dev_ptr) return RTHX_OK;
  CUG(cudaSetDevice(device_id));
  CUG(cudaIpcCloseMemHandle(dev_ptr));
  return RTHX_OK;
}

extern "C" int rthx_shared_free(int device_id, void* dev_ptr) {
  if (!dev_ptr) return RTHX_OK;
  CUG(cudaSetDevice(device_id));
  CUG(cudaFree(dev_ptr));
  return RTHX_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// device-side step flags for one-process-per-GPU runs: the ranks of a fused peer flush synchronise through 64-bit counters in
// the owner's memory (a release store over NVLink after the trace kernel, an acquire spin in front of the consumer) instead of
// a host-launched collective per step
// ---------------------------------------------------------------------------------------------------------------
namespace {
__global__ void flag_signal_kernel(unsigned long long* flag, unsigned long long value) {
  __threadfence_system();                                   // cumulative: everything the stream's earlier kernels wrote (the red.sys
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(flag), "l"(value) : "memory");   // flush of the rows) is visible before the flag
}
// lane i spins until flags[i] >= value; gives up after timeout_ns (a dead peer must not hang the GPU) and raises *err
__global__ void flag_wait_kernel(const unsigned long long* flags, int n, unsigned long long value, unsigned long long timeout_ns, unsigned long long* err) {
  unsigned long long t0, t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    for (;;) {
      unsigned long long v;
      asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(flags + i) : "memory");
      if (v >= value) break;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
      if (t - t0 > timeout_ns) { if (err) atomicAdd_system(err, 1ull); break; }   // the counter may live in the owner's (peer) memory
      __nanosleep(200);
    }
  }
  __threadfence_system();
}
}  // namespace

extern "C" int rthx_flag_signal(void* flag, uint64_t value, void* stream) {
  if (!flag) return fail(nullptr, RTHX_ERR_ARG, "rthx_flag_signal: NULL flag");
  flag_signal_kernel<<<1, 1, 0, (cudaStream_t)stream>>>((unsigned long long*)flag, (unsigned long long)value);
  CUG(cudaGetLastError());
  return RTHX_OK;
}

extern "C" int rthx_flag_wait(const void* flags, int n, uint64_t value, double timeout_s, void* err_flag, void* stream) {
  if (!flags || n < 1) return fail(nullptr, RTHX_ERR_ARG, "rthx_flag_wait: bad argument");
  const unsigned long long ns = (unsigned long long)((timeout_s > 0 ? timeout_s : 30.0) * 1e9);
  flag_wait_kernel<<<1, 32, 0, (cudaStream_t)stream>>>((const unsigned long long*)flags, n, (unsigned long long)value, ns, (unsigned long long*)err_flag);
  CUG(cudaGetLastError());
  return RTHX_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// sparse read-out of the resident counts
// ---------------------------------------------------------------------------------------------------------------
namespace rthx {
cudaError_t launch_row_nnz(const unsigned long long* c, int n_rows, int n_cols, size_t ld, int n_surf, int row_first, int row_stride, int* nnz,
                           unsigned long long* rowsum, unsigned long long* cross, cudaStream_t st);
cudaError_t launch_row_fill(const unsigned long long* c, int n_rows, int n_cols, size_t ld, const long long* row_ptr, const unsigned long long* rowsum, int* cols,
                            unsigned long long* vals, double* fvals, cudaStream_t st);
cudaError_t launch_csc_count(const unsigned long long* c, int n, size_t ld, int* partial, long long* colptr, cudaStream_t st);
cudaError_t launch_csc_fill(const unsigned long long* c, int n, size_t ld, const int* partial, const long long* colptr, const unsigned long long* rowsum,
                            int index_base, void* rowval, bool rowval_i64, unsigned long long* vals, double* fvals, cudaStream_t st);
cudaError_t launch_add_base(long long* p, int n, long long base, cudaStream_t st);
}  // namespace rthx

namespace {

// Device -> host copy of a result array on `stream`, blocking: `height` rows of `width` bytes (source pitch spitch, destination
// pitch dpitch; a flat array is one row).
//   * page-locked destination (cudaHostAlloc / cudaHostRegister, rthx_host_alloc): DMA.  With copy helpers registered
//     (rthx_set_copy_helpers: the handles of a multi-GPU trace on the other devices) a large copy is cut into one slice per device:
//     the owner's slice goes out over its own PCIe link, every other slice hops to its helper over NVLink (cudaMemcpyPeerAsync into
//     two 16 MB staging buffers, alternating streams) and leaves through THAT device's link — the 1.35 GB of cfg3's CSC arrays and
//     the 900 MB of F_smooth are PCIe-bound on one link (25 + 16 ms) and the other links are idle after a multi-GPU trace;
//   * pageable destination (a plain Julia / numpy array): through the handle's two pinned staging buffers in 32 MB pieces, the host
//     moving piece k-1 while piece k is in flight.
int copy_out_2d(rthx_handle* h, void* dst, size_t dpitch, const void* src_dev, size_t spitch, size_t width, size_t height, cudaStream_t stream) {
  if (width == 0 || height == 0) return RTHX_OK;
  cudaPointerAttributes pa;
  const bool pinned = cudaPointerGetAttributes(&pa, dst) == cudaSuccess && (pa.type == cudaMemoryTypeHost || pa.type == cudaMemoryTypeManaged);
  cudaGetLastError();
  const size_t bytes = width * height;
  auto direct = [&](size_t r0, size_t r1, cudaStream_t st) -> cudaError_t {
    if (r1 <= r0) return cudaSuccess;
    if (height == 1) return cudaMemcpyAsync(dst, src_dev, width, cudaMemcpyDeviceToHost, st);
    return cudaMemcpy2DAsync((char*)dst + r0 * dpitch, dpitch, (const char*)src_dev + r0 * spitch, spitch, width, r1 - r0, cudaMemcpyDeviceToHost, st);
  };
  const bool multi_link = pinned && !h->helpers.empty() && bytes >= (size_t(64) << 20) && std::getenv("RTHX_NO_COPY_HELPERS") == nullptr;
  if (pinned && !multi_link) {
    CU(h, direct(0, height, stream));
    CU(h, cudaStreamSynchronize(stream));
    return RTHX_OK;
  }
  if (multi_link) {
    // a flat array is re-cut into rows of 1 MB so that both shapes share the row-sliced code (the tail goes out with the owner's slice)
    size_t W = width, H = height, SP = spitch, DP = dpitch, tail = 0;
    if (height == 1) { W = SP = DP = size_t(1) << 20; H = width / W; tail = width - H * W; }
    const size_t n_links = h->helpers.size() + 1;
    const size_t chunk_rows = std::max<size_t>(1, (size_t(16) << 20) / SP);
    CU(h, cudaEventRecord(h->bev[16], stream));                       // the producer's work is done
    CU(h, cudaStreamWaitEvent(h->copy_stream, h->bev[16], 0));
    int rc = RTHX_OK;
    for (size_t l = 0; l < n_links && rc == RTHX_OK; ++l) {
      const size_t r0 = H * l / n_links, r1 = H * (l + 1) / n_links;
      if (l == 0) {
        if (r1 > r0) CU(h, cudaMemcpy2DAsync(dst, DP, src_dev, SP, W, r1 - r0, cudaMemcpyDeviceToHost, h->copy_stream));
        if (tail) CU(h, cudaMemcpyAsync((char*)dst + H * W, (const char*)src_dev + H * W, tail, cudaMemcpyDeviceToHost, h->copy_stream));
        continue;
      }
      rthx_handle* g = h->helpers[l - 1];
      auto enqueue = [&]() -> int {
        CU(g, cudaSetDevice(g->device));
        const size_t need = chunk_rows * SP;
        if (g->xfer_cap < need) {
          for (auto& xp : g->xfer) { if (xp) cudaFree(xp); xp = nullptr; }
          g->xfer_cap = 0;
          for (auto& xp : g->xfer) CU(g, cudaMalloc(&xp, need));
          g->xfer_cap = need;
        }
        CU(g, cudaStreamWaitEvent(g->stream, h->bev[16], 0));
        CU(g, cudaStreamWaitEvent(g->stream2, h->bev[16], 0));
        size_t k = 0;
        for (size_t a = r0; a < r1; a += chunk_rows, ++k) {
          const size_t b = std::min(r1, a + chunk_rows);
          cudaStream_t st = (k & 1) ? g->stream2 : g->stream;
          CU(g, cudaMemcpyPeerAsync(g->xfer[k & 1], g->device, (const char*)src_dev + a * SP, h->device, (b - a - 1) * SP + W, st));
          CU(g, cudaMemcpy2DAsync((char*)dst + a * DP, DP, g->xfer[k & 1], SP, W, b - a, cudaMemcpyDeviceToHost, st));
        }
        return RTHX_OK;
      };
      rc = enqueue();
      if (rc) h->err = g->err;
    }
    // wait for every link (also after an error, so that nothing is left in flight on the caller's buffers)
    for (rthx_handle* g : h->helpers) { cudaSetDevice(g->device); cudaStreamSynchronize(g->stream); cudaStreamSynchronize(g->stream2); }
    cudaSetDevice(h->device);
    if (rc) return rc;
    CU(h, cudaStreamSynchronize(h->copy_stream));
    return RTHX_OK;
  }
  // pageable destination
  if (bytes <= (size_t(1) << 20)) {
    CU(h, direct(0, height, stream));
    CU(h, cudaStreamSynchronize(stream));
    return RTHX_OK;
  }
  const size_t piece = size_t(32) << 20;
  if (h->stage_cap < piece) {
    for (auto& sp : h->stage) { if (sp) cudaFreeHost(sp); sp = nullptr; }
    h->stage_cap = 0;
    for (auto& sp : h->stage) CU(h, cudaMallocHost(&sp, piece));
    h->stage_cap = piece;
  }
  // pieces are whole rows (a flat array: 32 MB runs); the staging buffers hold them packed (pitch = width)
  const size_t rows_per_piece = height == 1 ? 1 : std::max<size_t>(1, piece / width);
  const size_t n_pieces = height == 1 ? (width + piece - 1) / piece : (height + rows_per_piece - 1) / rows_per_piece;
  auto piece_range = [&](size_t k, size_t& off_src, size_t& off_dst, size_t& w, size_t& rows) {
    if (height == 1) { off_src = off_dst = k * piece; w = std::min(piece, width - k * piece); rows = 1; }
    else { const size_t a = k * rows_per_piece; rows = std::min(rows_per_piece, height - a); off_src = a * spitch; off_dst = a * dpitch; w = width; }
  };
  auto unload = [&](size_t k) {
    size_t os, od, w, rows; piece_range(k, os, od, w, rows);
    if (rows == 1 || dpitch == w) parallel_memcpy((char*)dst + od, h->stage[k & 1], w * rows);
    else for (size_t r = 0; r < rows; ++r) std::memcpy((char*)dst + od + r * dpitch, (const char*)h->stage[k & 1] + r * w, w);
  };
  for (size_t k = 0; k < n_pieces; ++k) {
    size_t os, od, w, rows; piece_range(k, os, od, w, rows);
    if (rows == 1) CU(h, cudaMemcpyAsync(h->stage[k & 1], (const char*)src_dev + os, w, cudaMemcpyDeviceToHost, stream));
    else CU(h, cudaMemcpy2DAsync(h->stage[k & 1], w, (const char*)src_dev + os, spitch, w, rows, cudaMemcpyDeviceToHost, stream));
    CU(h, cudaEventRecord(h->cev[k & 1], stream));
    if (k >= 1) { CU(h, cudaEventSynchronize(h->cev[(k - 1) & 1])); unload(k - 1); }
  }
  CU(h, cudaEventSynchronize(h->cev[(n_pieces - 1) & 1]));
  unload(n_pieces - 1);
  return RTHX_OK;
}

int copy_out(rthx_handle* h, void* dst, const void* src_dev, size_t bytes, cudaStream_t stream) {
  return copy_out_2d(h, dst, bytes, src_dev, bytes, bytes, 1, stream);
}

// Row pass over the resident counts of `bin`: non-zeros and total per row, row pointers on the device, and the surface-gas
// cross-coupling chi of the row-normalised F (cross_coupling_chi, smoothExchangeFactors.jl:212-241).  After a sharded trace
// (emitter_world > 1: one row tile of a matrix too large to hold at once) the rows are those of the shard and chi is their share.
int prepare_rows(rthx_handle* h, int bin) {
  if (bin < 0 || bin >= h->last_trace_bins || (!h->counts_dev && !h->sparse_counts))
    return fail(h, RTHX_ERR_ARG, "counts: no resident counts for that bin (run rthx_trace_exchange with counts_out == NULL, rthx_trace_exchange_multi with counts_out == NULL, or rthx_trace_exchange_sparse first)");
  if (h->csr_bin == bin) return RTHX_OK;
  CU(h, cudaSetDevice(h->device));
  const int N = h->N, R = (int)h->last_trace_rows;
  if (h->csr_cap < (size_t)N + 1) {
    cudaFree(h->csr_nnz); cudaFree(h->csr_rowsum); cudaFree(h->csr_rowptr); cudaFree(h->csr_cross);
    h->csr_nnz = nullptr; h->csr_rowsum = nullptr; h->csr_rowptr = nullptr; h->csr_cross = nullptr; h->csr_cap = 0;
    CU(h, cudaMalloc(&h->csr_nnz, sizeof(int) * ((size_t)N + 1)));
    CU(h, cudaMalloc(&h->csr_rowsum, sizeof(unsigned long long) * ((size_t)N + 1)));
    CU(h, cudaMalloc(&h->csr_cross, sizeof(unsigned long long) * ((size_t)N + 1)));
    CU(h, cudaMalloc(&h->csr_rowptr, sizeof(long long) * ((size_t)N + 1)));
    h->csr_cap = (size_t)N + 1;
  }
  if (h->sparse_counts) {
    CU(h, rthx::tally_row_stats(h->sk_keys, h->sk_vals, h->sk_rowptr, h->last_trace_bins, bin, R, N, h->ns, h->last_rank, h->last_world, h->csr_nnz,
                                h->csr_rowsum, h->csr_cross, h->stream));
  } else {
    const unsigned long long* c = h->counts_dev + (size_t)bin * h->last_trace_rows * N;
    CU(h, rthx::launch_row_nnz(c, R, N, (size_t)N, h->ns, h->last_rank, h->last_world, h->csr_nnz, h->csr_rowsum, h->csr_cross, h->stream));
  }
  std::vector<int> nnz(std::max(R, 1));
  std::vector<unsigned long long> rowsum(std::max(R, 1)), cross(std::max(R, 1));
  if (R > 0) {
    CU(h, cudaMemcpyAsync(nnz.data(), h->csr_nnz, sizeof(int) * R, cudaMemcpyDeviceToHost, h->stream));
    CU(h, cudaMemcpyAsync(rowsum.data(), h->csr_rowsum, sizeof(unsigned long long) * R, cudaMemcpyDeviceToHost, h->stream));
    CU(h, cudaMemcpyAsync(cross.data(), h->csr_cross, sizeof(unsigned long long) * R, cudaMemcpyDeviceToHost, h->stream));
  }
  CU(h, cudaStreamSynchronize(h->stream));
  std::vector<long long> rp((size_t)R + 1, 0);
  double chi = 0.0;
  for (int i = 0; i < R; ++i) {
    rp[i + 1] = rp[i] + nnz[i];
    if (rowsum[i]) chi += (double)cross[i] / (double)rowsum[i];
  }
  CU(h, cudaMemcpyAsync(h->csr_rowptr, rp.data(), sizeof(long long) * ((size_t)R + 1), cudaMemcpyHostToDevice, h->stream));
  CU(h, cudaStreamSynchronize(h->stream));
  h->csr_bin = bin; h->csr_total = rp[R]; h->csr_chi = N ? chi / N : 0.0;
  return RTHX_OK;
}

}  // namespace

namespace rthx {
size_t sparse_sort_temp_bytes(int nnz, int n);
cudaError_t sparse_transpose(int n, int nnz, const long long* colptr, const int* rowval, const double* val, unsigned long long* keys,
                             unsigned long long* keys_sorted, double* val_sorted, long long* rptr, void* temp, size_t temp_bytes, cudaStream_t st);
}  // namespace rthx

namespace {
// Leading n x n block of the hashed tally's rows (bin `bin`, all emitters) as CSC in the sparse smoothing's scratch: colptr -> cp [n+1],
// rowval -> sp_rowval, F = count / row total over the block -> sp_val (the values rthx_counts_csc computes); *nnz_out its non-zeros.
// The CSR of the block is transposed by the radix sort of rthx_smooth_sparse (sparse_transpose), so rows ascend within each column.
// With counts != nullptr the count of every entry (as bits) is sorted along instead of F.  vec: 3 n scratch words.
int sparse_counts_to_csc(rthx_handle* h, int bin, int n, long long* cp, long long* rptr, void* vec, bool counts, long long* nnz_out) {
  unsigned long long* rowsum = reinterpret_cast<unsigned long long*>(vec);
  int* row_nnz = reinterpret_cast<int*>(rowsum + n);
  CU(h, rthx::tally_row_stats(h->sk_keys, h->sk_vals, h->sk_rowptr, h->last_trace_bins, bin, n, n, h->ns, 0, 1, row_nnz, rowsum, nullptr, h->stream));
  std::vector<int> rn((size_t)n);
  CU(h, cudaMemcpyAsync(rn.data(), row_nnz, sizeof(int) * (size_t)n, cudaMemcpyDeviceToHost, h->stream));
  CU(h, cudaStreamSynchronize(h->stream));
  std::vector<long long> rp((size_t)n + 1, 0);
  for (int i = 0; i < n; ++i) rp[i + 1] = rp[i] + rn[i];
  const long long nnz = rp[n];
  if (nnz > 0x7FFFFFFFll) return fail(h, RTHX_ERR_ARG, "sparse counts: more than 2^31 - 1 non-zeros in one column view");
  CU(h, cudaMemcpyAsync(rptr, rp.data(), sizeof(long long) * ((size_t)n + 1), cudaMemcpyHostToDevice, h->stream));
  const size_t nz1 = (size_t)std::max<long long>(nnz, 1);
  CU(h, ensure(&h->sp_rowval, &h->sp_rowval_cap, nz1));
  CU(h, ensure(&h->sp_val, &h->sp_val_cap, 2 * nz1));
  CU(h, ensure(&h->sp_keys, &h->sp_keys_cap, 2 * nz1));
  const size_t tmp_bytes = rthx::sparse_sort_temp_bytes((int)nnz, n);
  CU(h, ensure(reinterpret_cast<char**>(&h->sp_tmp), &h->sp_tmp_cap, tmp_bytes));
  CU(h, rthx::tally_row_fill(h->sk_keys, h->sk_vals, h->sk_rowptr, h->last_trace_bins, bin, n, n, rptr, rowsum, true, h->sp_rowval,
                             counts ? reinterpret_cast<unsigned long long*>(h->sp_val) : nullptr, counts ? nullptr : h->sp_val, h->stream));
  CU(h, rthx::sparse_transpose(n, (int)nnz, rptr, h->sp_rowval, h->sp_val, h->sp_keys, h->sp_keys + nz1, h->sp_val + nz1, cp, h->sp_tmp, tmp_bytes,
                               h->stream));
  *nnz_out = nnz;
  return RTHX_OK;
}

// rthx_counts_csc after a sparse trace: sorted transpose keys -> rowval (+ base), sorted values -> F_vals / vals
int counts_csc_sparse(rthx_handle* h, int bin, int index_base, int rowval_is_i64, int64_t* colptr, void* rowval, uint64_t* vals, double* F_vals) {
  const int N = h->N;
  CU(h, ensure(&h->csc_colptr, &h->csc_colptr_cap, (size_t)N + 1));
  const size_t need = (3 * (size_t)N + 1) * sizeof(unsigned long long);   // row pointers + row totals / non-zeros scratch
  if (h->csr_out_cap < need) {
    cudaFree(h->csr_out); h->csr_out = nullptr; h->csr_out_cap = 0;
    CU(h, cudaMalloc(&h->csr_out, need));
    h->csr_out_cap = need;
  }
  long long* rptr = reinterpret_cast<long long*>(h->csr_out);
  void* vec = rptr + (size_t)N + 1;
  long long nnz = 0;
  int rc = sparse_counts_to_csc(h, bin, N, h->csc_colptr, rptr, vec, false, &nnz);
  if (rc) return rc;
  if (F_vals && nnz && (rc = copy_out(h, F_vals, h->sp_val + std::max<long long>(nnz, 1), sizeof(double) * (size_t)nnz, h->stream))) return rc;
  if (vals) {                                                // the counts ride along a second sort of the same keys
    if ((rc = sparse_counts_to_csc(h, bin, N, h->csc_colptr, rptr, vec, true, &nnz))) return rc;
    if (nnz && (rc = copy_out(h, vals, h->sp_val + std::max<long long>(nnz, 1), sizeof(uint64_t) * (size_t)nnz, h->stream))) return rc;
  }
  const size_t nz1 = (size_t)std::max<long long>(nnz, 1);
  // the indices: low words of the sorted keys, written over the unsorted keys
  CU(h, rthx::tally_key_index(h->sp_keys + nz1, nnz, index_base, h->sp_keys, rowval_is_i64 != 0, h->stream));
  if (index_base) CU(h, rthx::launch_add_base(h->csc_colptr, N + 1, (long long)index_base, h->stream));
  if ((rc = copy_out(h, colptr, h->csc_colptr, sizeof(long long) * ((size_t)N + 1), h->stream))) return rc;
  if (nnz && (rc = copy_out(h, rowval, h->sp_keys, (rowval_is_i64 ? sizeof(long long) : sizeof(int)) * (size_t)nnz, h->stream))) return rc;
  CU(h, cudaStreamSynchronize(h->stream));
  return RTHX_OK;
}
}  // namespace

extern "C" int rthx_counts_nnz(rthx_handle* h, int bin, int64_t* nnz_out) {
  if (!h || !nnz_out) return RTHX_ERR_ARG;
  const int rc = prepare_rows(h, bin);
  if (rc) return rc;
  *nnz_out = h->csr_total;
  return RTHX_OK;
}

extern "C" int rthx_counts_stats(rthx_handle* h, int bin, int64_t* nnz_out, double* chi_out) {
  if (!h) return RTHX_ERR_ARG;
  const int rc = prepare_rows(h, bin);
  if (rc) return rc;
  if (nnz_out) *nnz_out = h->csr_total;
  if (chi_out) *chi_out = h->csr_chi;
  return RTHX_OK;
}

extern "C" int rthx_counts_csr(rthx_handle* h, int bin, int64_t* row_ptr, int32_t* cols, uint64_t* vals, double* F_vals) {
  if (!h || !row_ptr || !cols) return RTHX_ERR_ARG;
  int rc = prepare_rows(h, bin);
  if (rc) return rc;
  CU(h, cudaSetDevice(h->device));
  const int N = h->N;
  const size_t nnz = (size_t)h->csr_total;
  const size_t need = std::max<size_t>(1, nnz) * (sizeof(int) + sizeof(unsigned long long) + sizeof(double));
  if (h->csr_out_cap < need) {
    cudaFree(h->csr_out); h->csr_out = nullptr; h->csr_out_cap = 0;
    CU(h, cudaMalloc(&h->csr_out, need));
    h->csr_out_cap = need;
  }
  unsigned long long* d_vals = (unsigned long long*)h->csr_out;
  double* d_f = (double*)(d_vals + std::max<size_t>(1, nnz));
  int* d_cols = (int*)(d_f + std::max<size_t>(1, nnz));
  const int R = (int)h->last_trace_rows;
  if (h->sparse_counts) {
    CU(h, rthx::tally_row_fill(h->sk_keys, h->sk_vals, h->sk_rowptr, h->last_trace_bins, bin, R, N, h->csr_rowptr, h->csr_rowsum, false, d_cols, d_vals,
                               F_vals ? d_f : nullptr, h->stream));
  } else {
    const unsigned long long* c = h->counts_dev + (size_t)bin * h->last_trace_rows * N;
    CU(h, rthx::launch_row_fill(c, R, N, (size_t)N, h->csr_rowptr, h->csr_rowsum, d_cols, d_vals, F_vals ? d_f : nullptr, h->stream));
  }
  rc = copy_out(h, row_ptr, h->csr_rowptr, sizeof(long long) * ((size_t)R + 1), h->stream);
  if (rc) return rc;
  if (nnz) {
    if ((rc = copy_out(h, cols, d_cols, sizeof(int) * nnz, h->stream))) return rc;
    if (vals && (rc = copy_out(h, vals, d_vals, sizeof(unsigned long long) * nnz, h->stream))) return rc;
    if (F_vals && (rc = copy_out(h, F_vals, d_f, sizeof(double) * nnz, h->stream))) return rc;
  }
  CU(h, cudaStreamSynchronize(h->stream));
  return RTHX_OK;
}

extern "C" int rthx_counts_csc(rthx_handle* h, int bin, int index_base, int rowval_is_i64, int64_t* colptr, void* rowval, uint64_t* vals, double* F_vals) {
  if (!h || !colptr || !rowval || (index_base != 0 && index_base != 1)) return RTHX_ERR_ARG;
  if (h->last_trace_bins > 0 && (h->last_world != 1 || (int)h->last_trace_rows != h->N))
    return fail(h, RTHX_ERR_ARG, "counts_csc: the resident counts are the rows of a shard (emitter_world > 1); the column view needs the whole matrix");
  int rc = prepare_rows(h, bin);              // row totals for the normalisation, nnz for the buffer sizes
  if (rc) return rc;
  CU(h, cudaSetDevice(h->device));
  const int N = h->N;
  const size_t nnz = (size_t)h->csr_total, nz1 = std::max<size_t>(1, nnz);
  if (!rowval_is_i64 && (size_t)N + (size_t)index_base > 0x7FFFFFFFull) return fail(h, RTHX_ERR_ARG, "counts_csc: 32-bit row indices overflow");
  if (h->sparse_counts) { rc = counts_csc_sparse(h, bin, index_base, rowval_is_i64, colptr, rowval, vals, F_vals); if (rc) return rc; h->csc_bin = bin; return RTHX_OK; }
  const int n_tiles = (N + 63) / 64;
  CU(h, ensure(&h->csc_partial, &h->csc_partial_cap, (size_t)n_tiles * (size_t)N));
  CU(h, ensure(&h->csc_colptr, &h->csc_colptr_cap, (size_t)N + 1));
  const size_t need = nz1 * (sizeof(long long) + (vals ? sizeof(unsigned long long) : 0) + (F_vals ? sizeof(double) : 0));
  if (h->csr_out_cap < need) {
    cudaFree(h->csr_out); h->csr_out = nullptr; h->csr_out_cap = 0;
    CU(h, cudaMalloc(&h->csr_out, need));
    h->csr_out_cap = need;
  }
  long long* d_rows = (long long*)h->csr_out;                 // 8 bytes per entry reserved, holds int or long long indices
  unsigned long long* d_vals = vals ? (unsigned long long*)(d_rows + nz1) : nullptr;
  double* d_f = F_vals ? (double*)(d_rows + nz1 + (vals ? nz1 : 0)) : nullptr;
  const unsigned long long* c = h->counts_dev + (size_t)bin * h->last_trace_rows * N;
  CU(h, rthx::launch_csc_count(c, N, (size_t)N, h->csc_partial, h->csc_colptr, h->stream));
  CU(h, rthx::launch_csc_fill(c, N, (size_t)N, h->csc_partial, h->csc_colptr, h->csr_rowsum, index_base, d_rows, rowval_is_i64 != 0, d_vals, d_f, h->stream));
  if (index_base) CU(h, rthx::launch_add_base(h->csc_colptr, N + 1, (long long)index_base, h->stream));
  if ((rc = copy_out(h, colptr, h->csc_colptr, sizeof(long long) * ((size_t)N + 1), h->stream))) return rc;
  if (nnz) {
    if ((rc = copy_out(h, rowval, d_rows, (rowval_is_i64 ? sizeof(long long) : sizeof(int)) * nnz, h->stream))) return rc;
    if (vals && (rc = copy_out(h, vals, d_vals, sizeof(unsigned long long) * nnz, h->stream))) return rc;
    if (F_vals && (rc = copy_out(h, F_vals, d_f, sizeof(double) * nnz, h->stream))) return rc;
  }
  CU(h, cudaStreamSynchronize(h->stream));
  h->csc_bin = bin;
  return RTHX_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// reciprocity smoothing on the device
// ---------------------------------------------------------------------------------------------------------------
namespace rthx {
struct SmoothResult { int iters; double delta, delta_init; double ms_total, ms_per_iter; int launches; int converged; };
cudaError_t run_ap(const unsigned long long* src_counts, const double* src_F, const double* src_rs, size_t ld, const double* w_dev, int n, size_t ldx,
                   int max_iters, double target, double* X, double* rs, double* r, double* u, double* part, std::vector<double>& part_host, cudaStream_t st,
                   cudaEvent_t e0, cudaEvent_t e1, SmoothResult* out);
struct DykstraResult { int rounds; int pcg_iters; double delta; double ms; int launches; };
cudaError_t run_dykstra(const unsigned long long* src_counts, const double* src_F, size_t ld, const double* w_dev, int n, size_t ldx, int k_dykstra,
                        double* B, double* C, double* P, double* vec, cudaStream_t st, cudaEvent_t e0, cudaEvent_t e1, double** F_out, double** rs_out,
                        DykstraResult* out);
cudaError_t time_scale_pass(double* X, double* u, double* r, int n, size_t ldx, int reps, cudaStream_t st, cudaEvent_t e0, cudaEvent_t e1, double* ms_per_pass);
}  // namespace rthx

extern "C" int rthx_smooth_F(rthx_handle* h, int source, const void* src_host, int bin, int n, const double* w, int max_iters, double target,
                             int measure_pass, double* F_out, rthx_smooth_stats* st) {
  return rthx_smooth_DkAP(h, source, src_host, bin, n, w, 0, max_iters, target, measure_pass, F_out, st);
}

extern "C" int rthx_smooth_DkAP(rthx_handle* h, int source, const void* src_host, int bin, int n, const double* w, int k_dykstra, int max_iters,
                                double target, int measure_pass, double* F_out, rthx_smooth_stats* st) {
  if (!h) return RTHX_ERR_ARG;
  if (n < 1 || !w || !F_out || max_iters < 0 || k_dykstra < 0) return fail(h, RTHX_ERR_ARG, "smooth: bad argument");
  CU(h, cudaSetDevice(h->device));
  const size_t nn = (size_t)n * n;
  const unsigned long long* src_counts = nullptr;
  const double* src_F = nullptr;
  size_t ld = (size_t)n;
  if (source == RTHX_SMOOTH_FROM_LAST_TRACE) {
    if (h->sparse_counts)
      return fail(h, RTHX_ERR_ARG, "smooth: the resident counts are the sparse form of rthx_trace_exchange_sparse (smooth them with rthx_smooth_sparse)");
    if (bin < 0 || bin >= h->last_trace_bins || !h->counts_dev || n > h->N || h->last_world != 1 || (int)h->last_trace_rows != h->N)
      return fail(h, RTHX_ERR_ARG, "smooth: no resident counts for that bin (run rthx_trace_exchange on all emitters first)");
    src_counts = h->counts_dev + (size_t)bin * h->last_trace_rows * h->N;
    ld = (size_t)h->N;
  } else if (source == RTHX_SMOOTH_FROM_COUNTS || source == RTHX_SMOOTH_FROM_F) {
    if (!src_host) return fail(h, RTHX_ERR_ARG, "smooth: src_host is NULL");
    if (h->smooth_src_cap < nn * 8) {
      cudaFree(h->smooth_src); h->smooth_src = nullptr; h->smooth_src_cap = 0;
      CU(h, cudaMalloc(&h->smooth_src, nn * 8));
      h->smooth_src_cap = nn * 8;
    }
    CU(h, cudaMemcpyAsync(h->smooth_src, src_host, nn * 8, cudaMemcpyHostToDevice, h->stream));
    if (source == RTHX_SMOOTH_FROM_COUNTS) src_counts = (const unsigned long long*)h->smooth_src; else src_F = (const double*)h->smooth_src;
  } else {
    return fail(h, RTHX_ERR_ARG, "smooth: unknown source");
  }
  const size_t ldx = ((size_t)n + 15) & ~size_t(15);      // rows padded to 128 bytes
  h->smooth_n = 0;
  CU(h, ensure(&h->smooth_X, &h->smooth_cap, (size_t)n * ldx));
  CU(h, ensure(&h->smooth_vec, &h->smooth_vec_cap, (size_t)16 * ldx + 8));   // AP: w, rs, r, u, part; Dykstra: 10 vectors + 8 scalars
  double *w_dev = h->smooth_vec, *rs = w_dev + ldx, *r = rs + ldx, *u = r + ldx, *part = u + ldx;
  CU(h, cudaMemcpyAsync(w_dev, w, sizeof(double) * n, cudaMemcpyHostToDevice, h->stream));
  std::vector<double> part_host(n);
  rthx::SmoothResult res{};
  rthx::DykstraResult dres{};
  const double tgt = target > 0 ? target : 8 * 2.220446049250313e-16;
  const double* src_rs = nullptr;
  if (k_dykstra > 0) {
    // Dykstra rounds (DkAP, smoothExchangeFactors.jl:299-318) write into their own buffers; AP then builds X from the result
    const size_t mats = k_dykstra > 1 ? 3 : 1;
    CU(h, ensure(&h->dyk_buf, &h->dyk_cap, mats * (size_t)n * ldx));
    double* B = h->dyk_buf;
    double* Cb = mats > 1 ? B + (size_t)n * ldx : nullptr;
    double* Pb = mats > 1 ? Cb + (size_t)n * ldx : nullptr;
    double *Fd = nullptr, *rsd = nullptr;
    CU(h, rthx::run_dykstra(src_counts, src_F, ld, w_dev, n, ldx, k_dykstra, B, Cb, Pb, h->smooth_vec + 5 * ldx, h->stream, h->ev[2], h->ev[3], &Fd, &rsd, &dres));
    src_counts = nullptr; src_F = Fd; src_rs = rsd; ld = ldx;
  }
  CU(h, rthx::run_ap(src_counts, src_F, src_rs, ld, w_dev, n, ldx, max_iters, tgt, h->smooth_X, rs, r, u, part, part_host, h->stream, h->ev[0], h->ev[1], &res));
  {
    const int rcc = copy_out_2d(h, F_out, sizeof(double) * (size_t)n, h->smooth_X, sizeof(double) * ldx, sizeof(double) * (size_t)n, (size_t)n, h->stream);
    if (rcc) return rcc;
  }
  h->smooth_n = n; h->smooth_ldx = ldx;
  double pass_ms = 0;
  if (measure_pass) {
    std::vector<double> ones(ldx, 1.0);
    CU(h, cudaMemcpyAsync(u, ones.data(), sizeof(double) * ldx, cudaMemcpyHostToDevice, h->stream));
    CU(h, rthx::time_scale_pass(h->smooth_X, u, r, n, ldx, 20, h->stream, h->ev[0], h->ev[1], &pass_ms));
  }
  if (st) {
    st->iterations = res.iters; st->launches = res.launches; st->delta_init = res.delta_init; st->delta = res.delta;
    st->total_ms = res.ms_total; st->ms_per_iteration = res.ms_per_iter; st->pass_ms = pass_ms;
    st->pass_gbs = pass_ms > 0 ? 16.0 * (double)nn / (pass_ms * 1e-3) / 1e9 : 0.0;
    st->dykstra_rounds = dres.rounds; st->pcg_iterations = dres.pcg_iters; st->dykstra_delta = dres.rounds ? dres.delta : 0.0; st->dykstra_ms = dres.ms;
    st->launches += dres.launches;
    st->converged = res.converged; st->pad_ = 0;
  }
  return RTHX_OK;
}

namespace rthx {
size_t sparse_sort_temp_bytes(int nnz, int n);
cudaError_t sparse_transpose(int n, int nnz, const long long* colptr, const int* rowval, const double* val, unsigned long long* keys,
                             unsigned long long* keys_sorted, double* val_sorted, long long* rptr, void* temp, size_t temp_bytes, cudaStream_t st);
cudaError_t launch_x_count(int n, const long long* colptr, const int* rowval, const long long* rptr, const unsigned long long* keys_sorted, long long* xptr,
                           cudaStream_t st);
cudaError_t launch_x_fill(int n, const long long* colptr, const int* rowval, const double* val, const long long* rptr, const unsigned long long* keys_sorted,
                          const double* val_sorted, const double* w, long long* xptr, int* xcol, double* xval, cudaStream_t st);
cudaError_t run_ap_sparse(int n, long long nnz_f, long long nnz_x, const long long* xptr, const int* xcol, double* xval, const double* w, double* vec,
                          int max_iters, double target, cudaStream_t st, SmoothResult* out);
cudaError_t time_sparse_pass(int n, const long long* xptr, const int* xcol, double* xval, const double* w, double* vec, int reps, cudaStream_t st,
                             cudaEvent_t e0, cudaEvent_t e1, double* ms_per_pass);
cudaError_t launch_index_out(const int* col, long long nnz, int base, void* out, bool i64, cudaStream_t st);
}  // namespace rthx

extern "C" int rthx_smooth_sparse(rthx_handle* h, int source, int bin, int n, const int64_t* colptr, const int32_t* rowval, const double* nzval,
                                  const double* w, int max_iters, double target, int measure_pass, int64_t* nnz_out, rthx_smooth_stats* st) {
  if (!h) return RTHX_ERR_ARG;
  if (n < 1 || !w || !nnz_out || max_iters < 0) return fail(h, RTHX_ERR_ARG, "smooth_sparse: bad argument");
  long long nnz_f = 0;
  if (source == RTHX_SMOOTH_FROM_LAST_TRACE) {
    if (bin < 0 || bin >= h->last_trace_bins || (!h->counts_dev && !h->sparse_counts) || n > h->N || h->last_world != 1 || (int)h->last_trace_rows != h->N)
      return fail(h, RTHX_ERR_ARG, "smooth_sparse: no resident counts for that bin (run rthx_trace_exchange on all emitters first)");
  } else if (source == RTHX_SMOOTH_FROM_CSC) {
    // the whole matrix is checked here, before anything is uploaded: a bad index must never reach a kernel
    if (!colptr) return fail(h, RTHX_ERR_ARG, "smooth_sparse: colptr is NULL");
    if (colptr[0] != 0) return fail(h, RTHX_ERR_ARG, "smooth_sparse: colptr[0] must be 0 (0-based CSC)");
    for (int j = 0; j < n; ++j)
      if (colptr[j + 1] < colptr[j]) return fail(h, RTHX_ERR_ARG, "smooth_sparse: colptr decreases at column " + std::to_string(j));
    nnz_f = colptr[n];
    if (nnz_f > 0x7FFFFFFFll) return fail(h, RTHX_ERR_ARG, "smooth_sparse: more than 2^31 - 1 non-zeros");
    if (nnz_f > 0 && (!rowval || !nzval)) return fail(h, RTHX_ERR_ARG, "smooth_sparse: rowval / nzval is NULL");
    for (int j = 0; j < n; ++j)
      for (long long p = colptr[j]; p < colptr[j + 1]; ++p)
        if (rowval[p] < 0 || rowval[p] >= n || (p > colptr[j] && rowval[p] <= rowval[p - 1]))
          return fail(h, RTHX_ERR_ARG, "smooth_sparse: rowval out of [0, n) or not strictly ascending in column " + std::to_string(j));
  } else {
    return fail(h, RTHX_ERR_ARG, "smooth_sparse: unknown source");
  }
  CU(h, cudaSetDevice(h->device));
  h->smooth_n = 0;                 // a dense F_smooth left by rthx_smooth_F is no longer the handle's smoothing result
  h->sparse_n = 0;
  const size_t n1 = (size_t)n + 1;
  CU(h, ensure(&h->sp_ptr, &h->sp_ptr_cap, 3 * n1));
  CU(h, ensure(&h->sp_vec, &h->sp_vec_cap, 5 * (size_t)n + 8));
  long long *cp = h->sp_ptr, *rptr = cp + n1, *xptr = rptr + n1;
  double* w_dev = h->sp_vec;
  double* vec = w_dev + n;                                     // r | u | u' | part | scalars
  CU(h, cudaMemcpyAsync(w_dev, w, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, h->stream));
  CU(h, cudaEventRecord(h->ev[0], h->stream));
  if (source == RTHX_SMOOTH_FROM_LAST_TRACE && h->sparse_counts) {
    // the hashed tally's rows cropped to n, F = count / row total over the crop, transposed to CSC (same values and order as below)
    int rc = sparse_counts_to_csc(h, bin, n, cp, rptr, vec + n, false, &nnz_f);
    if (rc) return rc;
    const size_t nz1 = (size_t)std::max<long long>(nnz_f, 1);
    CU(h, rthx::tally_key_index(h->sp_keys + nz1, nnz_f, 0, h->sp_rowval, false, h->stream));
    if (nnz_f) CU(h, cudaMemcpyAsync(h->sp_val, h->sp_val + nz1, sizeof(double) * (size_t)nnz_f, cudaMemcpyDeviceToDevice, h->stream));
  } else if (source == RTHX_SMOOTH_FROM_LAST_TRACE) {
    // F = counts / row total over the crop, compacted to CSC by the read-out kernels of rthx_counts_csc
    const unsigned long long* c = h->counts_dev + (size_t)bin * h->last_trace_rows * h->N;
    const size_t ld = (size_t)h->N;
    unsigned long long* rowsum = reinterpret_cast<unsigned long long*>(vec + n);   // u and u' are free until the iteration
    int* row_nnz = reinterpret_cast<int*>(vec + 2 * (size_t)n);
    CU(h, ensure(&h->csc_partial, &h->csc_partial_cap, (size_t)((n + 63) / 64) * (size_t)n));
    CU(h, rthx::launch_row_nnz(c, n, n, ld, h->ns, 0, 1, row_nnz, rowsum, nullptr, h->stream));
    CU(h, rthx::launch_csc_count(c, n, ld, h->csc_partial, cp, h->stream));
    CU(h, cudaMemcpyAsync(&nnz_f, cp + n, sizeof(long long), cudaMemcpyDeviceToHost, h->stream));
    CU(h, cudaStreamSynchronize(h->stream));
    if (nnz_f > 0x7FFFFFFFll) return fail(h, RTHX_ERR_ARG, "smooth_sparse: more than 2^31 - 1 non-zeros");
    CU(h, ensure(&h->sp_rowval, &h->sp_rowval_cap, (size_t)std::max<long long>(nnz_f, 1)));
    CU(h, ensure(&h->sp_val, &h->sp_val_cap, 2 * (size_t)std::max<long long>(nnz_f, 1)));
    CU(h, rthx::launch_csc_fill(c, n, ld, h->csc_partial, cp, rowsum, 0, h->sp_rowval, false, nullptr, h->sp_val, h->stream));
  } else {
    CU(h, ensure(&h->sp_rowval, &h->sp_rowval_cap, (size_t)std::max<long long>(nnz_f, 1)));
    CU(h, ensure(&h->sp_val, &h->sp_val_cap, 2 * (size_t)std::max<long long>(nnz_f, 1)));
    CU(h, cudaMemcpyAsync(cp, colptr, sizeof(long long) * n1, cudaMemcpyHostToDevice, h->stream));
    if (nnz_f > 0) {
      CU(h, cudaMemcpyAsync(h->sp_rowval, rowval, sizeof(int) * (size_t)nnz_f, cudaMemcpyHostToDevice, h->stream));
      CU(h, cudaMemcpyAsync(h->sp_val, nzval, sizeof(double) * (size_t)nnz_f, cudaMemcpyHostToDevice, h->stream));
    }
  }
  // transpose (CSR of F), then X on the union pattern
  const size_t nz1 = (size_t)std::max<long long>(nnz_f, 1);
  CU(h, ensure(&h->sp_keys, &h->sp_keys_cap, 2 * nz1));
  const size_t tmp_bytes = rthx::sparse_sort_temp_bytes((int)nnz_f, n);
  CU(h, ensure(reinterpret_cast<char**>(&h->sp_tmp), &h->sp_tmp_cap, tmp_bytes));
  double* val_sorted = h->sp_val + nz1;
  unsigned long long* keys_sorted = h->sp_keys + nz1;
  CU(h, rthx::sparse_transpose(n, (int)nnz_f, cp, h->sp_rowval, h->sp_val, h->sp_keys, keys_sorted, val_sorted, rptr, h->sp_tmp, tmp_bytes, h->stream));
  CU(h, rthx::launch_x_count(n, cp, h->sp_rowval, rptr, keys_sorted, xptr, h->stream));
  long long nnz_x = 0;
  CU(h, cudaMemcpyAsync(&nnz_x, xptr + n, sizeof(long long), cudaMemcpyDeviceToHost, h->stream));
  CU(h, cudaStreamSynchronize(h->stream));
  CU(h, ensure(&h->sp_xcol, &h->sp_xcol_cap, (size_t)std::max<long long>(nnz_x, 1)));
  CU(h, ensure(&h->sp_xval, &h->sp_xval_cap, (size_t)std::max<long long>(nnz_x, 1)));
  CU(h, rthx::launch_x_fill(n, cp, h->sp_rowval, h->sp_val, rptr, keys_sorted, val_sorted, w_dev, xptr, h->sp_xcol, h->sp_xval, h->stream));
  rthx::SmoothResult res{};
  const double tgt = target > 0 ? target : 8 * 2.220446049250313e-16;
  CU(h, rthx::run_ap_sparse(n, nnz_f, nnz_x, xptr, h->sp_xcol, h->sp_xval, w_dev, vec, max_iters, tgt, h->stream, &res));
  CU(h, cudaEventRecord(h->ev[1], h->stream));
  CU(h, cudaStreamSynchronize(h->stream));
  float ms = 0;
  CU(h, cudaEventElapsedTime(&ms, h->ev[0], h->ev[1]));
  h->sparse_n = n; h->sparse_nnz = nnz_x;
  *nnz_out = nnz_x;
  double pass_ms = 0;
  if (measure_pass) CU(h, rthx::time_sparse_pass(n, xptr, h->sp_xcol, h->sp_xval, w_dev, vec, 20, h->stream, h->ev[0], h->ev[1], &pass_ms));
  if (st) {
    std::memset(st, 0, sizeof(*st));
    st->iterations = res.iters; st->launches = res.launches; st->delta_init = res.delta_init; st->delta = res.delta;
    st->total_ms = ms; st->ms_per_iteration = res.iters > 0 ? ms / res.iters : 0.0; st->pass_ms = pass_ms;
    st->pass_gbs = pass_ms > 0 ? (20.0 * (double)nnz_x + 8.0 * (double)n1) / (pass_ms * 1e-3) / 1e9 : 0.0;
    st->converged = res.converged;
  }
  return RTHX_OK;
}

extern "C" int rthx_smooth_sparse_csc(rthx_handle* h, int index_base, int rowval_is_i64, int64_t* colptr, void* rowval, double* nzval) {
  if (!h) return RTHX_ERR_ARG;
  if (!colptr || !rowval || !nzval || (index_base != 0 && index_base != 1)) return fail(h, RTHX_ERR_ARG, "smooth_sparse_csc: bad argument");
  if (h->sparse_n < 1) return fail(h, RTHX_ERR_ARG, "smooth_sparse_csc: no sparse F_smooth on this handle (run rthx_smooth_sparse first)");
  CU(h, cudaSetDevice(h->device));
  const int n = h->sparse_n;
  const long long nnz = h->sparse_nnz;
  const long long* xptr = h->sp_ptr + 2 * ((size_t)n + 1);
  int rc = copy_out(h, colptr, xptr, sizeof(long long) * ((size_t)n + 1), h->stream);
  if (rc) return rc;
  if (index_base) for (int i = 0; i <= n; ++i) colptr[i] += index_base;
  if (nnz > 0) {
    const void* idx = h->sp_xcol;
    if (index_base || rowval_is_i64) {         // the key buffers (>= 16 bytes per entry of F, >= 8 per entry of F_smooth) are free now
      CU(h, rthx::launch_index_out(h->sp_xcol, nnz, index_base, h->sp_keys, rowval_is_i64 != 0, h->stream));
      idx = h->sp_keys;
    }
    if ((rc = copy_out(h, rowval, idx, (rowval_is_i64 ? sizeof(long long) : sizeof(int)) * (size_t)nnz, h->stream))) return rc;
    if ((rc = copy_out(h, nzval, h->sp_xval, sizeof(double) * (size_t)nnz, h->stream))) return rc;
  }
  CU(h, cudaStreamSynchronize(h->stream));
  return RTHX_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// rthx_solve_grey: (I - diag(coeff) F') j = h by restarted GMRES on the device (kernels in rthx_solve.cu)
// ---------------------------------------------------------------------------------------------------------------
extern "C" int rthx_solve_grey(rthx_handle* h, const rthx_solve_args* a, double* j_out, double* g_out, rthx_solve_stats* st) {
  if (!h) return RTHX_ERR_ARG;
  if (!a || !j_out || a->n < 1 || !a->coeff || !a->rhs) return fail(h, RTHX_ERR_ARG, "solve: bad argument");
  CU(h, cudaSetDevice(h->device));
  const int n = a->n;
  const int m = std::max(1, std::min(a->memory > 0 ? a->memory : 50, n));
  const int max_iters = a->max_iters > 0 ? a->max_iters : 2 * n;
  const double rtol = a->rtol > 0 ? a->rtol : 1e-12;
  const double atol = a->atol >= 0 ? a->atol : 1.4901161193847656e-08;   // sqrt(eps(Float64))
  const size_t nl = ((size_t)n + 15) & ~size_t(15);
  rthx::SolveMatrix A;
  if (a->source == RTHX_SOLVE_FROM_LAST_SMOOTH) {
    if (h->smooth_n != n || !h->smooth_X) return fail(h, RTHX_ERR_ARG, "solve: no resident F_smooth of that size (run rthx_smooth_F on this handle first)");
    A.kind = 0; A.dense = h->smooth_X; A.ld = h->smooth_ldx;
  } else if (a->source == RTHX_SOLVE_FROM_DENSE) {
    if (!a->F_dense || (a->layout != RTHX_ROW_MAJOR && a->layout != RTHX_COL_MAJOR)) return fail(h, RTHX_ERR_ARG, "solve: F_dense is NULL or unknown layout");
    CU(h, ensure(&h->solve_mat, &h->solve_mat_cap, (size_t)n * nl));
    CU(h, cudaMemsetAsync(h->solve_mat, 0, sizeof(double) * (size_t)n * nl, h->stream));      // row padding must read as zeros
    CU(h, cudaMemcpy2DAsync(h->solve_mat, sizeof(double) * nl, a->F_dense, sizeof(double) * (size_t)n, sizeof(double) * (size_t)n, (size_t)n,
                            cudaMemcpyHostToDevice, h->stream));
    A.kind = a->layout == RTHX_ROW_MAJOR ? 0 : 1; A.dense = h->solve_mat; A.ld = nl;
  } else if (a->source == RTHX_SOLVE_FROM_CSC) {
    if (!a->colptr || (!a->rowval && a->colptr[n] > 0) || (!a->nzval && a->colptr[n] > 0)) return fail(h, RTHX_ERR_ARG, "solve: CSC arrays missing");
    const long long nnz = a->colptr[n];
    if (nnz < 0 || a->colptr[0] != 0) return fail(h, RTHX_ERR_ARG, "solve: colptr must be 0-based and non-decreasing");
    // one buffer: nzval [nnz] doubles | colptr [n+1] i64 | rowval [nnz] i32
    const size_t need = (size_t)std::max<long long>(nnz, 1) + (size_t)(n + 1) + ((size_t)std::max<long long>(nnz, 1) + 1) / 2 + 4;
    CU(h, ensure(&h->solve_mat, &h->solve_mat_cap, need));
    double* nz = h->solve_mat;
    long long* cp = reinterpret_cast<long long*>(nz + std::max<long long>(nnz, 1));
    int* rv = reinterpret_cast<int*>(cp + (n + 1));
    if (nnz > 0) {
      CU(h, cudaMemcpyAsync(nz, a->nzval, sizeof(double) * (size_t)nnz, cudaMemcpyHostToDevice, h->stream));
      CU(h, cudaMemcpyAsync(rv, a->rowval, sizeof(int) * (size_t)nnz, cudaMemcpyHostToDevice, h->stream));
    }
    CU(h, cudaMemcpyAsync(cp, a->colptr, sizeof(long long) * (size_t)(n + 1), cudaMemcpyHostToDevice, h->stream));
    A.kind = 2; A.colptr = cp; A.rowval = rv; A.nzval = nz; A.nnz = nnz;
  } else {
    return fail(h, RTHX_ERR_ARG, "solve: unknown source");
  }
  const size_t vec = rthx::solve_vec_doubles(nl, m);
  const size_t part = A.kind == 0 ? rthx::solve_part_doubles(n, A.ld) : 0;
  CU(h, ensure(&h->solve_buf, &h->solve_cap, vec + part));
  CU(h, cudaMemsetAsync(h->solve_buf, 0, sizeof(double) * vec, h->stream));
  double* coeff_dev = h->solve_buf + (size_t)(m + 4) * nl;     // layout of run_gmres: V[(m+1)] | w | x | r | coeff | rhs | d
  double* rhs_dev = coeff_dev + nl;
  CU(h, cudaMemcpyAsync(coeff_dev, a->coeff, sizeof(double) * n, cudaMemcpyHostToDevice, h->stream));
  CU(h, cudaMemcpyAsync(rhs_dev, a->rhs, sizeof(double) * n, cudaMemcpyHostToDevice, h->stream));
  rthx::SolveResult res{};
  CU(h, rthx::run_gmres(A, n, nl, m, max_iters, rtol, atol, h->solve_buf, h->solve_buf + vec, j_out, g_out, h->stream, h->ev[0], h->ev[1], &res));
  double mv_ms = 0;
  if (a->measure_pass) CU(h, rthx::time_matvec(A, n, nl, m, h->solve_buf, h->solve_buf + vec, 20, h->stream, h->ev[0], h->ev[1], &mv_ms));
  if (st) {
    std::memset(st, 0, sizeof(*st));
    st->iterations = res.iterations; st->restarts = res.restarts; st->launches = res.launches; st->converged = res.converged; st->matvecs = res.matvecs;
    st->residual = res.residual; st->rhs_norm = res.rhs_norm; st->total_ms = res.total_ms; st->matvec_bytes = res.matvec_bytes;
    st->matvec_ms = mv_ms; st->matvec_gbs = mv_ms > 0 ? (double)res.matvec_bytes / (mv_ms * 1e-3) / 1e9 : 0.0;
  }
  return RTHX_OK;
}

extern "C" int rthx_measure_fp64_peak(rthx_handle* h, double* tflops) {
  if (!h || !tflops) return RTHX_ERR_ARG;
  CU(h, cudaSetDevice(h->device));
  const int threads = 256, blocks = h->prop.multiProcessorCount * 8, iters = 1 << 15;
  if (!h->peak_dev) CU(h, cudaMalloc(&h->peak_dev, sizeof(double) * (size_t)threads * blocks));
  CU(h, launch_fp64_peak(h->peak_dev, blocks, threads, 1024, h->stream));  // warm-up
  double best = 0;
  for (int rep = 0; rep < 3; ++rep) {
    CU(h, cudaEventRecord(h->ev[0], h->stream));
    CU(h, launch_fp64_peak(h->peak_dev, blocks, threads, iters, h->stream));
    CU(h, cudaEventRecord(h->ev[1], h->stream));
    CU(h, cudaStreamSynchronize(h->stream));
    float ms = 0;
    CU(h, cudaEventElapsedTime(&ms, h->ev[0], h->ev[1]));
    const double flops = 2.0 * 8.0 * (double)iters * threads * blocks;
    best = std::max(best, flops / (ms * 1e-3) / 1e12);
  }
  *tflops = best;
  return RTHX_OK;
}
