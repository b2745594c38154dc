// rthx_kernels.cu — sm_100a kernels of the exchange-factor tracer.
//
// K1 trace_exchange_kernel fuses the four stages of the path for one (emitter row, band, ray chunk) per block:
//   (1) emitter sampling, one thread per ray, counter-based Philox4x32-10 keyed by (seed | ray id, emitter, band)
//       — emitSurfaceRay2D.jl:1-27 + lambertSample2D.jl:1-11, emitVolumeRay2D.jl:1-33;
//   (2) first-interaction traversal (traceRay.jl:20-147 with distToSurface2D.jl:2-18 and the point location of
//       findFace2D.jl:1-101, replaced by an analytic lattice inverse on verified affine sub-meshes);
//   (3) tally into a per-block shared-memory u32 histogram of the block's source row, flushed with red.add.u64
//       into the global count matrix (parallelRayTracing.jl:104,124,144-146);
//   (4) optional RayRecorder output of origin / endpoint (parallelRayTracing.jl:108,120-123,135-138).
// No tensor cores: the path is branchy FP64 geometry + integer RNG + integer atomics, not a contraction.
#include <climits>
#include "rthx_internal.h"

#include <math_constants.h>

namespace rthx {

// ------------------------------------------------------------------------------------------------------------
// RNG: Philox4x32-10 and the uniform conversions of the rthx.h contract
// ------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    k.x += 0x9E3779B9u;
    k.y += 0xBB67AE85u;
  }
  return c;
}

// Same generator with the 10 round keys precomputed on the host (TraceParams::rk, parameter bank): the key schedule
// disappears from the instruction stream and the LOP3s take the keys as c[0][..] operands.
__device__ __forceinline__ uint4 philox4x32_10_rk(uint4 c, const uint32_t* __restrict__ rk) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ rk[2 * r], lo1, hi0 ^ c.w ^ rk[2 * r + 1], lo0);
  }
  return c;
}

// Uniforms by mantissa injection.  The subtrahends live in the kernel parameter bank (p.k_*), so each conversion is
// two integer ops + one DADD with a constant-bank operand instead of a 64-bit immediate materialised by two UMOVs.
//   u52: ((x >> 12) + 0.5) * 2^-52, x = hi:lo   = [1,2) - (1 - 2^-53), exact
//   u32: (w + 0.5) * 2^-32                      = [1,2) - (1 - 2^-33), exact
//   u23: ((w >> 9) + 0.5) * 2^-23 (Float32)     = [1,2) - (1 - 2^-24), exact
__device__ __forceinline__ double u52(uint32_t lo, uint32_t hi, double k_u52) {
  return __hiloint2double((int)(0x3FF00000u | (hi >> 12)), (int)((hi << 20) | (lo >> 12))) - k_u52;
}
__device__ __forceinline__ double u32d(uint32_t w, double k_u32) {
  return __hiloint2double((int)(0x3FF00000u | (w >> 12)), (int)(w << 20)) - k_u32;
}
__device__ __forceinline__ float u23(uint32_t w) {
  return __uint_as_float(0x3F800000u | (w >> 9)) - 0.999999940395355224609375f;  // 1 - 2^-24
}

// ------------------------------------------------------------------------------------------------------------
// geometry primitives
// ------------------------------------------------------------------------------------------------------------
// distToSurface2D.jl:2-18 on a coarse face: smallest positive u_i = ((v_i - p)·n_i)/(d·n_i) over edges with
// |d·n_i| >= 1e-10, first index on ties.  Branch-free: the argmin runs on cross-multiplied fractions (one division
// instead of nv; u_i > 0 <=> num_i*den_i > 0), and the unused 4th edge of a triangle has a zero normal, so it can
// never pass the |den| test.  Ties/rounding differ from the reference only on a set of measure ~1e-16.
__device__ __forceinline__ double dist_to_coarse(const CoarseDev& f, double px, double py, double dx, double dy, double eps, int& k) {
  double bn = 1.0, bd = 0.0;  // best |num| / |den|; bd == 0 <=> no candidate yet (any candidate beats it)
  int bk = 0;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const double nx = f.nx[i], ny = f.ny[i];
    const double den = dx * nx + dy * ny;
    const double num = (f.vx[i] - px) * nx + (f.vy[i] - py) * ny;
    const double an = fabs(num), ad = fabs(den);
    const bool better = (ad >= eps) & (num * den > 0.0) & (an * bd < bn * ad);
    bn = better ? an : bn;
    bd = better ? ad : bd;
    bk = better ? i : bk;
  }
  k = bk;
  return bd > 0.0 ? bn / bd : CUDART_INF;
}

// ---- FAST-path math -------------------------------------------------------------------------------------------
// Coefficients live in __constant__ memory so DFMA takes them as constant-bank operands (a 64-bit immediate costs
// two UMOVs per use in SASS; libdevice's log/cospi spend ~40 issue slots per ray on those alone).
__constant__ double c_sinpi[9] = {  // sin(pi z) = z * P(z^2), |z| <= 1/2, max abs error 2.2e-16 (Chebyshev fit, mpmath)
    0x1.921fb54442d18p+1, -0x1.4abbce625be52p+2, 0x1.466bc6775aa7dp+1, -0x1.32d2cce627c86p-1, 0x1.5078348551854p-4,
    -0x1.e3074dfaf87afp-8, 0x1.e8f3675ee37ddp-12, -0x1.6f7acdb8f6580p-16, 0x1.9d462020fcc78p-21};

// sqrt(x) and a/b for well-scaled positive normal operands (variates in (0,1), geometric ratios): MUFU seed + Newton,
// without libdevice's special-case branch (which splits the basic block and blocks instruction interleaving).
// Accurate to <= 2 ulp (sqrt) / 1 ulp (div); neither is used where x or b can be 0, Inf or subnormal.
__device__ __forceinline__ double sqrt_pos(double x) {
  double y;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));   // MUFU.RSQ64H: ~2^-20 relative
  const double g = x * y;                                   // sqrt(x) sqrt(1 - e),  e = 1 - x y^2
  const double e = fma(-g, y, 1.0);
  return fma(fma(e, 0.375, 0.5), g * e, g);                 // g (1 + e/2 + 3 e^2/8): ~2^-58; 5 FP64 instructions
}
// a / |b|: the magnitude is taken on the high word (integer pipe); MUFU.RCP64H reads only that word
__device__ __forceinline__ double div_pos_abs(double a, double b) {
  const double ba = __hiloint2double(__double2hiint(b) & 0x7FFFFFFF, __double2loint(b));
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(ba));
  r = fma(r, fma(-ba, r, 1.0), r);
  const double q = a * r;
  return fma(r, fma(-ba, q, a), q);
}
__device__ __forceinline__ double div_pos(double a, double b) {
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(b));     // MUFU.RCP64H: ~2^-20 relative
  r = fma(r, fma(-b, r, 1.0), r);                           // ~2^-40
  const double q = a * r;
  return fma(r, fma(-b, q, a), q);                          // residual correction: <= 1 ulp
}

// The same polynomial for the argument y = R - 1/2 (what the mantissa injection delivers in ONE DADD): with z' = |y| - 1/4 = z/2,
// sin(pi z) = z' * P'(z'^2), P'_k = 2 * 4^k * P_k.  Scaling by powers of two is exact, so the result is bit-identical to
// cos2pi_unit(R) — it only drops the DFMA 2R-1 and the two IMAD.MOVs that materialise its 2.0.
__constant__ double c_sinpi2[9] = {
    0x1.921fb54442d18p+1 * 0x1p1, -0x1.4abbce625be52p+2 * 0x1p3, 0x1.466bc6775aa7dp+1 * 0x1p5, -0x1.32d2cce627c86p-1 * 0x1p7,
    0x1.5078348551854p-4 * 0x1p9, -0x1.e3074dfaf87afp-8 * 0x1p11, 0x1.e8f3675ee37ddp-12 * 0x1p13, -0x1.6f7acdb8f6580p-16 * 0x1p15,
    0x1.9d462020fcc78p-21 * 0x1p17};
__device__ __forceinline__ double cos2pi_centered(double y) {
  const double z = fabs(y) - 0.25;
  const double w = z * z;
  double p = c_sinpi2[8];
#pragma unroll
  for (int k = 7; k >= 0; --k) p = fma(p, w, c_sinpi2[k]);
  return z * p;
}
// 2 cos(2 pi R): the same coefficients times two (exact), for sin(theta) = 2 sqrt(R (1 - R))
__constant__ double c_sinpi4[9] = {
    0x1.921fb54442d18p+1 * 0x1p2, -0x1.4abbce625be52p+2 * 0x1p4, 0x1.466bc6775aa7dp+1 * 0x1p6, -0x1.32d2cce627c86p-1 * 0x1p8,
    0x1.5078348551854p-4 * 0x1p10, -0x1.e3074dfaf87afp-8 * 0x1p12, 0x1.e8f3675ee37ddp-12 * 0x1p14, -0x1.6f7acdb8f6580p-16 * 0x1p16,
    0x1.9d462020fcc78p-21 * 0x1p18};
__device__ __forceinline__ double cos2pi_centered_x2(double y) {
  const double z = fabs(y) - 0.25;
  const double w = z * z;
  double p = c_sinpi4[8];
#pragma unroll
  for (int k = 7; k >= 0; --k) p = fma(p, w, c_sinpi4[k]);
  return z * p;
}
// u32 uniform minus 1/2, exact: [1,2) - (3/2 - 2^-33)
__device__ __forceinline__ double u32d_centered(uint32_t w, double k_u32c) {
  return __hiloint2double((int)(0x3FF00000u | (w >> 12)), (int)(w << 20)) - k_u32c;
}

// cos(2 pi R) for R in (0,1): with x = 2R - 1 in (-1,1), cos(2 pi R) = -cos(pi x) = sin(pi (|x| - 1/2)); branch-free.
__device__ __forceinline__ double cos2pi_unit(double R) {
  const double z = fabs(fma(R, 2.0, -1.0)) - 0.5;
  const double w = z * z;
  double p = c_sinpi[8];
#pragma unroll
  for (int k = 7; k >= 0; --k) p = fma(p, w, c_sinpi[k]);
  return z * p;
}

// -log(x) by table: x = 2^e m, m in [1,2) falls in one of 256 intervals with midpoint c_i; with r = m/c_i - 1 (|r| <= 2^-9)
//   log x = e ln2 + log c_i + log1p(r),   log1p(r) = r - r^2/2 + r^3/3 - r^4/4 + r^5/5   (truncation r^6/6 < 2^-56)
// 8 FP64 instructions instead of ~30 for the fdlibm form (FP64 instructions are the expensive ones of this kernel: the pipe
// takes a warp every other cycle).  Absolute error <= 1e-15 on -log x <= 37 (relative <= 1e-16 except within 1e-10 of x = 1,
// where the free path itself is ~1e-10 and an absolute 1e-16 is immaterial).  The (1/c_i, log c_i) pairs (tools/gen_logtab.py)
// are staged into shared memory per block (4 KB).
#include "rthx_logtab.h"

__constant__ double c_l1p[4] = {0x1.999999999999ap-3 /* 1/5 */, 0x1.5555555555555p-2 /* 1/3 */, 0x1.62e42fefa39efp-1 /* ln 2 */, 0.0};

__device__ __forceinline__ double neg_log_table(double x, const double2* __restrict__ tab) {
  const int hi = __double2hiint(x), lo = __double2loint(x);
  const int e = (hi >> 20) - 1023;
  const double m = __hiloint2double((hi & 0x000FFFFF) | 0x3FF00000, lo);
  const double2 t = tab[(hi >> 12) & (LOGTAB_N - 1)];
  const double r = fma(m, t.x, -1.0);
  const double P = fma(r, fma(r, fma(r, c_l1p[0], -0.25), c_l1p[1]), -0.5);
  return -(fma((double)e, c_l1p[2], t.y) + fma(r * r, P, r));
}

// distToSurface2D on a coarse face, FAST path.  The emission / crossing point is inside the face, so edge i can
// only be hit when the ray moves outward through it (d·n_i >= 1e-10) with a positive plane distance h_i - p·n_i.
//   quads (parallelograms): slab form — edges 0/2 share the normal n0, edges 1/3 the normal n1: two dot products per
//                           axis instead of four per edge, and the sign of d·n picks the edge of each pair;
//   triangles             : three edges.
// The argmin runs on cross-multiplied fractions (first index on ties), one division at the end.
__device__ __forceinline__ double dist_quad(const CoarseDev& f, double px, double py, double dx, double dy, double eps, int& k) {
  const double n0x = f.nx[0], n0y = f.ny[0], n1x = f.nx[1], n1y = f.ny[1];
  const double den0 = dx * n0x + dy * n0y, q0 = px * n0x + py * n0y;
  const double den1 = dx * n1x + dy * n1y, q1 = px * n1x + py * n1y;
  const bool p0 = den0 > 0.0, p1 = den1 > 0.0;
  const double an0 = p0 ? f.h[0] - q0 : q0 - f.h[2], ad0 = fabs(den0);
  const double an1 = p1 ? f.h[1] - q1 : q1 - f.h[3], ad1 = fabs(den1);
  const int e0 = p0 ? 0 : 2, e1 = p1 ? 1 : 3;
  const bool ok0 = (ad0 >= eps) & (an0 > 0.0), ok1 = (ad1 >= eps) & (an1 > 0.0);
  const double l = an0 * ad1, r = an1 * ad0;
  const bool take0 = ok0 & (!ok1 | (l < r) | ((l == r) & (e0 < e1)));
  k = take0 ? e0 : e1;
  const double an = take0 ? an0 : an1, ad = take0 ? ad0 : ad1;
  return (ok0 | ok1) ? div_pos(an, ad) : CUDART_INF;
}

__device__ __forceinline__ double dist_fast(const CoarseDev& f, double px, double py, double dx, double dy, double eps, int& k) {
  if (f.kind == KIND_AFFINE_QUAD) return dist_quad(f, px, py, dx, dy, eps, k);
  double bn = 1.0, bd = 0.0;
  int bk = 0;
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const double nx = f.nx[i], ny = f.ny[i];
    const double den = dx * nx + dy * ny;
    const double num = f.h[i] - (px * nx + py * ny);
    const bool better = (den >= eps) & (num > 0.0) & (num * bd < bn * den);
    bn = better ? num : bn;
    bd = better ? den : bd;
    bk = better ? i : bk;
  }
  k = bk;
  return bd > 0.0 ? div_pos(bn, bd) : CUDART_INF;
}

// Generic locator.  One 96-byte record per polygon (rthx_api.cu, face_record), read with 32-byte loads — the generic kernel is
// bound by the L1 data pipe, which moves one 32-byte sector per lane and load instruction whatever the access width:
//   rec = { vx[4], vy[4], {vertex count, normal-orientation bits, surface id of walls 0..3, -} }
// (a triangle repeats its first vertex in slot 3: the zero-length edge never straddles py, so four edges serve both kinds).
struct __align__(32) Quad64 { double a, b, c, d; };
__device__ __forceinline__ Quad64 ldg256(const double* __restrict__ ptr) {          // LDG.E.256 (sm_100)
  Quad64 r;
  asm("ld.global.nc.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(r.a), "=d"(r.b), "=d"(r.c), "=d"(r.d) : "l"(ptr));
  return r;
}

// distToSurface2D on the polygon of a record, index of the nearest edge only (the wall of a fine cell a ray ends on,
// traceRay.jl:51): u_i = ((v_i - p).n_i)/(d.n_i) over the edges with |d.n_i| >= 1e-10 and u_i > 0, first index on ties.
// The argmin runs on cross-multiplied fractions — no division — and on the UNNORMALISED outward normals a_i = +-(ey, -ex) of the
// edges (v_i -> v_i+1), built from the vertices: u_i is a ratio, the factor |e_i| cancels, and the threshold reads
// (d.a_i)^2 >= 1e-20 |e_i|^2.  No per-polygon normal arrays are read: vertices + tail are three sectors.
// Returns the wall index; `surf` gets the surface id of that wall (-1: not a solid wall).
__device__ __forceinline__ int wall_of_rec(const double* __restrict__ rec, double px, double py, double dx, double dy, int& surf) {
  const Quad64 X = ldg256(rec), Y = ldg256(rec + 4), T = ldg256(rec + 8);
  const double vx[4] = {X.a, X.b, X.c, X.d}, vy[4] = {Y.a, Y.b, Y.c, Y.d};
  const int nv = __double2loint(T.a), bits = __double2hiint(T.a);
  double bn = 1.0, bd = 0.0;   // best |num| / |den|; bd == 0: no candidate yet
  int bi = 0;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int j = (i + 1) & 3;                                                       // (slot 3 of a triangle is vertex 0)
    const double ex = vx[j] - vx[i], ey = vy[j] - vy[i];
    const bool flip = (bits >> i) & 1;
    const double ax = flip ? -ey : ey, ay = flip ? ex : -ex;
    const double den = dx * ax + dy * ay;
    const double num = (vx[i] - px) * ax + (vy[i] - py) * ay;
    const double an = fabs(num), ad = fabs(den);
    const bool better = (i < nv) & (den * den >= 1e-20 * (ex * ex + ey * ey)) & (num * den > 0.0) & (an * bd < bn * ad);
    bn = better ? an : bn; bd = better ? ad : bd; bi = better ? i : bi;
  }
  surf = bi == 0 ? __double2loint(T.b) : (bi == 1 ? __double2hiint(T.b) : (bi == 2 ? __double2loint(T.c) : __double2hiint(T.c)));
  return bi;
}

// pointInPolygonFast2D, findFace2D.jl:77-101 (crossing number) on the vertices of a record.
// The crossing test "px < xi + (xj-xi)/(yj-yi) (py-yi)" is evaluated without the division:
//   t = (px-xi)(yj-yi) - (xj-xi)(py-yi) has the sign of (px - ix)(yj-yi), so the edge is crossed iff t (yj-yi) < 0
// — exact except for a point within rounding of an edge.  The CPU oracle keeps the reference's form; the exact-parity tests bound
// the difference (<= 2e-6 of the rays).
__device__ __forceinline__ bool point_in_rec(const double* __restrict__ rec, double px, double py) {
  const Quad64 X = ldg256(rec), Y = ldg256(rec + 4);
  const double vx[4] = {X.a, X.b, X.c, X.d}, vy[4] = {Y.a, Y.b, Y.c, Y.d};
  unsigned inside = 0u;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int j = (i + 3) & 3;
    const double xi = vx[i], yi = vy[i], xj = vx[j], yj = vy[j];
    const bool straddle = (yi > py) != (yj > py);
    const double dyv = yj - yi;
    const double t = fma(px - xi, dyv, -((xj - xi) * (py - yi)));
    const bool crossed = straddle & (t != 0.0) & (((__double2hiint(t) ^ __double2hiint(dyv)) < 0));
    inside ^= crossed ? 1u : 0u;
  }
  return inside != 0u;
}

// findFaceUniformGrid2D, findFace2D.jl:2-27: the face of set `set` that contains (px, py) — local face index or -1.
// The reference scans a bucket of ~9 bounding-box candidates for the first face passing the crossing-number test.  Which face
// contains a point does not depend on the grid, so the device's grid (rthx_grid.h, build_grid) is ~12x finer per axis, lists only the
// polygons that really meet the bucket, and marks the buckets that lie wholly inside one face:
//   trip 1: the set's grid (three uniform 16-byte loads) and the bucket's 16-byte entry {code, a, b, c};
//           code 0 (84 % of the buckets of a regular mesh): the answer is a — one sector per location, no vertex test;
//   trip 2: code k >= 1: crossing-number test on candidates a, b, c (k > 3: bucket_cand[a..a+k)) in ascending face order, first hit.
// (The bbox-prefilter fallback of findFace2D.jl:30-45 can only succeed where the bucket scan succeeds, up to rounding of the bucket
// index on a set of measure zero; it is restated in the CPU oracle and omitted here.)
// History: round 1 walked the reference's bucket serially (10 of 32 lanes busy, two L2 trips per candidate, 3.1e9 rays/s on cfg3);
// round 2 first tested all bounding boxes of a bucket into a bit mask (1.2e10), then put box + vertices of every bucket entry in one
// 128-byte record (1.37e10: ncu showed the L1 data pipe 98.7 % busy with ~19 sectors per ray, hence this layout).
__device__ __noinline__ int find_face_generic(const TraceParams& p, int set, double px, double py) {
  const double2* fs2 = reinterpret_cast<const double2*>(p.sets + set);
  const double2 org = __ldg(fs2), inv = __ldg(fs2 + 1);
  const int4 g = __ldg(reinterpret_cast<const int4*>(fs2 + 2));        // nx, ny, bucket_off, poly_base
  const double fi = floor((px - org.x) * inv.x), fj = floor((py - org.y) * inv.y);
  if (!(fi >= 0.0 && fi < (double)g.x && fj >= 0.0 && fj < (double)g.y)) return -1;
  const int4 e = __ldg(p.bucket_ent + (g.z + (int)fi + (int)fj * g.x));
  if (e.x == 0) return e.y;
  const double* recs = p.face_rec + 12 * (size_t)g.w;
  if (e.x <= 3) {
    if (e.x >= 1 && point_in_rec(recs + 12 * (size_t)e.y, px, py)) return e.y;
    if (e.x >= 2 && point_in_rec(recs + 12 * (size_t)e.z, px, py)) return e.z;
    if (e.x >= 3 && point_in_rec(recs + 12 * (size_t)e.w, px, py)) return e.w;
    return -1;
  }
  for (int k = 0; k < e.x; ++k) {
    const int f = __ldg(p.bucket_cand + e.y + k);
    if (point_in_rec(recs + 12 * (size_t)f, px, py)) return f;
  }
  return -1;
}

// Fine-cell location by the analytic lattice inverse: returns the local fine index or -1.
__device__ __forceinline__ int locate_affine(const TraceParams& p, const CoarseDev& cf, double px, double py) {
  const double rx = px - cf.ax, ry = py - cf.ay;
  const double s = rx * cf.g1x + ry * cf.g1y, t = rx * cf.g2x + ry * cf.g2y;
  const int n = __double2int_rd(s), m = __double2int_rd(t);   // NaN -> 0, caught by the range test on s,t below
  if (!((s >= 0.0) & (t >= 0.0) & (n < cf.Nx) & (m < cf.Ny))) return -1;
  const int cell = n + m * cf.Nx;
  if (cf.kind == KIND_AFFINE_QUAD) return cell;
  return __ldg(p.lattice + cf.lat_off + cell);
}

// the same for a face known to be a parallelogram lattice (fine index = n + m Nx, meshQuad.jl:139,151)
__device__ __forceinline__ int locate_quad(const CoarseDev& cf, double px, double py) {
  const double rx = px - cf.ax, ry = py - cf.ay;
  const double s = rx * cf.g1x + ry * cf.g1y, t = rx * cf.g2x + ry * cf.g2y;
  const int n = __double2int_rd(s), m = __double2int_rd(t);
  if (!((s >= 0.0) & (t >= 0.0) & (n < cf.Nx) & (m < cf.Ny))) return -1;
  return n + m * cf.Nx;
}

template <bool FAST>
__device__ __forceinline__ int locate_fine(const TraceParams& p, const CoarseDev& cf, int c, int kind, double px, double py) {
  if (!FAST && kind == KIND_GENERIC) return find_face_generic(p, 1 + c, px, py);
  return locate_affine(p, cf, px, py);
}

// ------------------------------------------------------------------------------------------------------------
// Flush of a block's row histogram into the count matrix.
//   matrix on this GPU   : one red.global.add.u64 per non-zero bin (several chunks of a row add up in place);
//   matrix in peer memory (one-process-per-GPU / multi-device gather, rows of different GPUs are disjoint): nothing on the wire is
//       atomic.  A block that owns its whole row (row_chunks == 1) writes it out with plain coalesced stores; otherwise the chunks
//       of a row add up in a LOCAL staging row first and the chunk that arrives last (per-row ticket) hands the finished row over.
//       NVLink then carries exactly 8 N bytes per row, overlapped with the tracing of the other rows — with system-scope reductions
//       per chunk it carried row_chunks times that in 8-byte atomics, which at 8 GPUs x 15 chunks doubled the kernel time.
// The kernels keep their plain red.add flush inline for a matrix on their own GPU and call this (out of line) only for a matrix in
// peer memory.  Everything it needs is recomputed from blockIdx and the parameter bank, so that it keeps no register alive across
// the ray loop (the SQ loop sits exactly at the 64 registers of 4 resident blocks per SM).
// `ticket`: one free word of the block's dynamic shared memory (the upper half of the emitter block's last slot) — a static
// __shared__ variable would eat into the opt-in maximum the kernels are configured for.
__device__ __noinline__ void handover_row_hist(const TraceParams& p, const uint32_t* hist, unsigned int* ticket) {
  const int N = p.N;
  const unsigned t1 = blockIdx.x / (unsigned)p.row_chunks;
  const int bi = (int)(t1 % (unsigned)p.n_bins);
  const int y = p.y_offset + (int)(t1 / (unsigned)p.n_bins);
  const int e = p.emitter_rank + y * p.emitter_world;
  unsigned long long* dst = p.peer_counts + ((size_t)bi * N + e) * (size_t)N;
  if (p.row_chunks == 1) {
    for (int i = threadIdx.x; i < N; i += blockDim.x) dst[i] = (unsigned long long)hist[i];
    return;
  }
  unsigned long long* count_row = p.counts + ((size_t)bi * p.n_owned + y) * (size_t)N;      // local compact staging row
  for (int i = threadIdx.x; i < N; i += blockDim.x) {
    const uint32_t v = hist[i];
    if (v) atomicAdd(&count_row[i], (unsigned long long)v);
  }
  __threadfence();                                       // this chunk's reductions are visible before its ticket is drawn
  __syncthreads();
  if (threadIdx.x == 0) *ticket = atomicAdd(&p.row_done[(size_t)bi * p.n_owned + y], 1u);
  __syncthreads();
  if (*ticket == (unsigned int)p.row_chunks - 1u) {      // last chunk of the row: every other chunk has fenced and drawn before
    __threadfence();
    for (int i = threadIdx.x; i < N; i += blockDim.x) dst[i] = __ldcg(&count_row[i]);
  }
}

// ------------------------------------------------------------------------------------------------------------
// Hashed row tally (HASH instances of K1, rthx_trace_exchange_sparse): the block's row lives in a shared-memory open-addressing
// table — keys absorber + 1 (0 = empty), u32 counts, 2^sk_slots_log2 slots, linear probing — instead of a u32[N] histogram or a
// dense u64 row.  Rays are traced in block-synchronous rounds of blockDim.x; before a round the table is flushed if it could pass
// half full during the round, so an insert always finds a slot.  A flush appends the occupied slots as (row key << 32 | column,
// count) pairs to a global buffer (one atomic per block reserves the space) and clears the table.  When the buffer is full the
// block raises the overflow flag and stops: the host re-runs that group of rows split in two.
// Table layout: keys [S] u32 | counts [S] u32 | occupied u32 | fill u32 | base u64.
// ------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void hash_insert(uint32_t* tab, int log2s, int absorber) {
  const uint32_t mask = (1u << log2s) - 1u, key = (uint32_t)absorber + 1u;
  uint32_t s = (key * 0x9E3779B1u) >> (32 - log2s);
  for (;;) {
    const uint32_t prev = atomicCAS(&tab[s], 0u, key);
    if (prev == 0u || prev == key) {
      atomicAdd(&tab[(mask + 1u) + s], 1u);
      if (prev == 0u) atomicAdd(&tab[2 * (mask + 1u)], 1u);
      return;
    }
    s = (s + 1u) & mask;
  }
}

// Block-uniform: every thread calls it at the same point.  Returns false when the pair buffer is full (the block must stop).
__device__ __noinline__ bool hash_flush(const TraceParams& p, uint32_t* tab, unsigned long long row_key) {
  const uint32_t S = 1u << p.sk_slots_log2;
  uint32_t* occ = tab + 2 * S;
  unsigned long long* base = reinterpret_cast<unsigned long long*>(tab + 2 * S + 2);
  __syncthreads();                                       // the round's inserts are complete
  const uint32_t n = *occ;
  if (n == 0) return true;
  if (threadIdx.x == 0) {
    const unsigned long long b = atomicAdd(&p.sk_ctl[0], (unsigned long long)n);
    if (b + n > p.sk_cap) { atomicExch(&p.sk_ctl[1], 1ull); *base = ~0ull; }
    else { *base = b; atomicAdd(&p.sk_ctl[2], 1ull); }
    occ[1] = 0u;
  }
  __syncthreads();
  const unsigned long long b = *base;
  if (b == ~0ull) return false;
  const int lane = threadIdx.x & 31;
  for (uint32_t i0 = 0; i0 < S; i0 += blockDim.x) {      // ballot + popc compaction, one shared-memory atomic per warp
    const uint32_t i = i0 + threadIdx.x;
    const uint32_t k = i < S ? tab[i] : 0u;
    const unsigned m = __ballot_sync(0xffffffffu, k != 0u);
    uint32_t w = 0;
    if (lane == 0 && m) w = atomicAdd(&occ[1], (uint32_t)__popc(m));
    w = __shfl_sync(0xffffffffu, w, 0);
    if (k) {
      const unsigned long long d = b + w + __popc(m & ((1u << lane) - 1u));
      p.sk_keys[d] = (row_key << 32) | (unsigned long long)(k - 1u);
      p.sk_cnt[d] = tab[S + i];
      tab[i] = 0u; tab[S + i] = 0u;
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) *occ = 0u;
  __syncthreads();
  return true;
}

// ------------------------------------------------------------------------------------------------------------
// K1: fused emit + trace + tally (+ record)
//   HIST_SMEM: per-block shared-memory row histogram (else direct global atomics, N > ~57 k elements)
//   HASH     : hashed row tally into (row, column, count) pairs (see above; HIST_SMEM == false): trace_exchange_hash_kernel
//   FAST     : every coarse face is a verified affine lattice with a complete neighbour table and the coarse
//              descriptors fit in shared memory -> no generic locator code in the kernel at all
//   MINB     : minimum resident blocks per SM the register allocation is bounded for
// ------------------------------------------------------------------------------------------------------------
// Block-uniform emitter description, kept in shared memory (broadcast LDS) instead of ~24 registers per thread.
//   surface emitter: [0,1] p1, [2,3] edge p2-p1, [4,5] xVecLocal (unit edge), [6,7] yVecLocal (left normal)
//   volume emitter : [0..5] triangle ABC as (V0, V1-V0, V2-V0), [6..11] triangle CDA likewise, [14] area(ABC)/volume
//   both           : [12,13] cell midPoint
constexpr int EM_DOUBLES = 16;

//   MULTI    : RTHX_MULTI_BOUNCE event loop
//   SQ       : the whole domain is ONE parallelogram coarse face (every square / rectangular enclosure): its descriptor
//              is read from the kernel-parameter bank (FP64 instructions take c[0][..] operands: no LDS, no address
//              arithmetic), there is no coarse-face loop and no per-face kind dispatch
template <bool HIST_SMEM, bool FAST, int MINB, bool MULTI, bool SQ>
__global__ void __launch_bounds__(256, MINB) trace_exchange_kernel(const __grid_constant__ TraceParams p) {
  constexpr bool HASH = false;
#include "rthx_trace_body.cuh"
}

// the same kernel with the hashed row tally (FIRST_INTERACTION, no histogram; the host rejects MULTI_BOUNCE before a launch)
template <bool FAST>
__global__ void __launch_bounds__(256, 2) trace_exchange_hash_kernel(const __grid_constant__ TraceParams p) {
  constexpr bool HIST_SMEM = false, MULTI = false, SQ = false, HASH = true;
#include "rthx_trace_body.cuh"
}

// ------------------------------------------------------------------------------------------------------------
// K1-SQ: the fused kernel for domains that are ONE parallelogram coarse face (every square / rectangular enclosure:
// cfg1-4).  Same arithmetic as the SQ branch of trace_exchange_kernel; what differs is the code shape:
//   * the three block-uniform decisions — surface or volume emitter, uniform or cell-wise beta, recorder on or off —
//     are taken ONCE, outside the ray loop, into eight specialised loop bodies.  Each loop keeps only its own
//     constants live, so the uniform-register file no longer overflows (the single shared loop spent ~40 of 327 warp
//     instructions per 32 rays on LDCU / R2UR / MOV.SPILL / UMOV / S2UR constant shuffling) and carries no dead branches;
//   * 32-bit loop counter relative to the block's first ray;
//   * the lattice inverse and the emission nudge use pre-folded constants (s = p.g1 + c1 instead of (p - a).g1; p(1-nudge) +
//     mid nudge instead of p + (mid - p) nudge): 4 FP64 instructions fewer, results equal to 1 ulp of the coordinates.
// ------------------------------------------------------------------------------------------------------------
// The triangle selector of emitVolumeRay2D.jl:7 as an integer compare:  (w + 1/2) 2^-32 < a  <=>  w < ceil(a 2^32 - 1/2)  (all
// operations exact in double for a 2^32 < 2^52).  Returns the largest word that still selects triangle ABC; a >= 1 (triangular
// cells: a = 2) selects it always.  (a <= 2^-33, a degenerate ABC, would select it for w = 0 only instead of never.)
__device__ __forceinline__ uint32_t selector_threshold(double a) {
  double t = ceil(a * 4294967296.0 - 0.5);
  t = fmin(fmax(t, 1.0), 4294967296.0);
  return (uint32_t)((unsigned long long)t - 1ull);
}

// Block prologue of the SQ / queue kernels (one thread): the emitter description with the emission nudge
// p + (mid - p) nu (emitSurfaceRay2D.jl:10, emitVolumeRay2D.jl:22) folded into the geometry, so that no per-ray instruction is
// spent on it:  surface  p = [(1-nu) p1 + nu mid] + R [(1-nu) (p2 - p1)];  volume  p = [(1-nu) V0 + nu mid] + a1 [(1-nu) (V1-V0)] + ...
// (positions equal the unfolded form to 1 ulp).
//   surface emitter: [0,1] origin, [2,3] edge, [4,5] xVecLocal (unit edge), [6,7] yVecLocal (left normal)
//   volume emitter : [0..5] triangle ABC as (V0, V1-V0, V2-V0), [6..11] triangle CDA likewise, [14] area(ABC)/volume,
//                    [15] (as u32) the integer triangle selector
__device__ __forceinline__ void stage_emitter_folded(const TraceParams& p, int g, int wall, double* s_em) {
  const int em_nv = p.poly_nv[g];
  const double* vx = p.poly_vx + 4 * g;
  const double* vy = p.poly_vy + 4 * g;
  const double omn = 1.0 - p.nudge, mxn = p.cell_mid[2 * g] * p.nudge, myn = p.cell_mid[2 * g + 1] * p.nudge;
  if (wall >= 0) {
    const int j = (wall + 1 == em_nv) ? 0 : wall + 1;
    const double ex = vx[j] - vx[wall], ey = vy[j] - vy[wall];
    const double len = sqrt(ex * ex + ey * ey);
    s_em[0] = fma(vx[wall], omn, mxn); s_em[1] = fma(vy[wall], omn, myn); s_em[2] = ex * omn; s_em[3] = ey * omn;
    s_em[4] = ex / len; s_em[5] = ey / len;
    s_em[6] = -(ey / len); s_em[7] = ex / len;
  } else {
    s_em[0] = vx[0]; s_em[1] = vy[0]; s_em[2] = vx[1] - vx[0]; s_em[3] = vy[1] - vy[0]; s_em[4] = vx[2] - vx[0]; s_em[5] = vy[2] - vy[0];
    s_em[6] = vx[2]; s_em[7] = vy[2]; s_em[8] = vx[3] - vx[2]; s_em[9] = vy[3] - vy[2]; s_em[10] = vx[0] - vx[2]; s_em[11] = vy[0] - vy[2];
    s_em[14] = em_nv == 3 ? 2.0 : 0.5 * (vx[0] * (vy[1] - vy[2]) + vx[1] * (vy[2] - vy[0]) + vx[2] * (vy[0] - vy[1])) / p.cell_volume[g];
    reinterpret_cast<uint32_t*>(s_em + 15)[0] = selector_threshold(s_em[14]);
    for (int t = 0; t < 12; t += 6) {
      s_em[t] = fma(s_em[t], omn, mxn); s_em[t + 1] = fma(s_em[t + 1], omn, myn);
      for (int q = 2; q < 6; ++q) s_em[t + q] *= omn;
    }
  }
}

// Stage 1 for one ray from its eight Philox words: emission point (nudge included), in-plane direction and the free-path
// variate.  dy_m is a double of magnitude |dy| and dy_hi the high word of dy: the volume sampler holds -dy = 2R - 1 and leaves
// the negation to the consumers (an operand modifier in FP64 instructions, one xor where the sign bit is read).
template <bool SURF>
__device__ __forceinline__ void emit_ray_folded(const TraceParams& p, const double* __restrict__ s_em, uint32_t sel_thr, const uint4& w0, const uint4& w1,
                                                double& px, double& py, double& dx, double& dy, double& dy_m, int& dy_hi, double& R_S) {
  if (SURF) {
    const double R = u32d(w0.x, p.k_u32);
    px = fma(s_em[2], R, s_em[0]);
    py = fma(s_em[3], R, s_em[1]);
    // lambertSample2D: Float32 variates / sqrt / square, the rest in Float64
    const float cosT = __fsqrt_rn(u23(w0.y));
    const float cos2 = __fmul_rn(cosT, cosT);
    const double sinT = sqrt_pos(1.0 - (double)cos2);
    const double xdir = sinT * cos2pi_centered((double)u23(w0.z) - 0.5);
    const double zdir = (double)cosT;
    dx = s_em[4] * xdir + s_em[6] * zdir;
    dy = s_em[5] * xdir + s_em[7] * zdir;
    dy_m = dy;
    dy_hi = __double2hiint(dy);
    R_S = u52(w1.x, w1.y, p.k_u52);
  } else {
    const double R1 = u32d(w0.x, p.k_u32), R2 = u32d(w0.y, p.k_u32);
    const double sq = sqrt_pos(R1);
    // triangle ABC or CDA (emitVolumeRay2D.jl:7): (w + 1/2) 2^-32 < area(ABC)/area  <=>  w <= thr, an integer compare
    const double* tri = s_em + ((w0.z <= sel_thr) ? 0 : 6);
    const double a2 = sq * R2, a1 = sq - a2;
    px = fma(a2, tri[4], fma(a1, tri[2], tri[0]));
    py = fma(a2, tri[5], fma(a1, tri[3], tri[1]));
    // theta = acos(1 - 2R): with c = R - 1/2 (one DADD from the mantissa injection), cos = -2c and sin = 2 sqrt(1/4 - c^2);
    // 1/4 - c^2 = R (1 - R) exactly, so one fma rounds to the same double as the product did
    const double c = __hiloint2double((int)(0x3FF00000u | (w1.y >> 12)), (int)((w1.y << 20) | (w1.x >> 12))) - p.k_u52c;
    dx = sqrt_pos(fma(-c, c, 0.25)) * cos2pi_centered_x2(u32d_centered(w0.w, p.k_u32c));
    dy_m = c + c;
    dy = -dy_m;
    dy_hi = __double2hiint(dy_m) ^ (int)0x80000000;
    R_S = u52(w1.z, w1.w, p.k_u52);
  }
}

struct SqBlock {            // block-uniform state of one (emitter row, band, chunk)
  const double* s_em;       // emitter description (shared memory, EM_DOUBLES)
  const double2* s_log;     // -log table (shared memory)
  uint32_t* hist;           // row histogram (shared memory)
  const double* beta_band;  // per-cell beta of the band (non-uniform bins)
  double inv_beta_u;
  uint32_t sel_thr;         // volume emitters: take triangle ABC iff Philox word <= sel_thr
  const double* omega_band; // MULTI_BOUNCE: scattering albedo per cell of the band
  const double* eps_band;   // MULTI_BOUNCE: emissivity per surface of the band
  uint32_t e, cw;
  int64_t ray0;             // ray id of the block's first ray
  uint32_t n_rays;          // rays of this block
  size_t rec_base;          // recorder slot of the block's first ray
};

// Fine-cell index on the single lattice.  One unsigned compare per axis covers both ends of the range: a negative
// coordinate floors to a negative integer (out of range as unsigned), an overflow saturates to INT_MIN/INT_MAX; s, t are finite
// here (the advance length is finite whenever this is reached), so no NaN -> 0 alias can occur.
template <bool AXIS>
__device__ __forceinline__ int locate_sq(const TraceParams& p, double px, double py) {
  const CoarseDev& cf = p.face0;
  const double s = AXIS ? fma(px, cf.g1x, p.sq_lc1) : fma(px, cf.g1x, fma(py, cf.g1y, p.sq_lc1));
  const double t = AXIS ? fma(py, cf.g2y, p.sq_lc2) : fma(px, cf.g2x, fma(py, cf.g2y, p.sq_lc2));
  const int n = __double2int_rd(s), m = __double2int_rd(t);
  return (((unsigned)n < (unsigned)cf.Nx) & ((unsigned)m < (unsigned)cf.Ny)) ? n + m * cf.Nx : -1;
}

__device__ __forceinline__ double flip_sign(double x, int sign_src_hi) {   // x with its sign bit xor-ed by the sign bit of a high word
  return __hiloint2double(__double2hiint(x) ^ (sign_src_hi & (int)0x80000000), __double2loint(x));
}

// distToSurface2D on the single parallelogram, slab form about the centre lines: with t_a = p.n_a - cen_a, the plane distance
// along the pair of edges with normal +-n_a is  hw_a - sign(d.n_a) t_a  (edge a if d.n_a > 0, edge a+2 otherwise).  Signs are
// read from the high words (integer pipe), the argmin runs on cross-multiplied fractions, one division at the end.
// AXIS: n0 = (0, +-1), n1 = (+-1, 0): d.n0 = +-dy, p.n0 = +-py — the four dot products disappear (bit-identical results).
// Returns false when no edge lies ahead (the reference's u = Inf).
template <bool AXIS>
__device__ __forceinline__ bool dist_sq(const TraceParams& p, double px, double py, double dx, double dy, double dy_m, int dy_hi, double& u, int& k) {
  const CoarseDev& f = p.face0;
  double d0, d1, tf0, tf1;                        // d.n0, d.n1 up to sign (only |.| is used), sign(d.n_a) (p.n_a - cen_a)
  int s0, s1;                                     // high words carrying the sign of d.n0, d.n1
  if (AXIS) {
    // dy_m: any double of magnitude |dy|, dy_hi: the high word of dy (a caller that holds -dy passes it with the flipped word
    // and saves the negation: only |d.n0| and its sign are used here)
    s0 = dy_hi ^ (int)p.sq_flip0; s1 = __double2hiint(dx) ^ (int)p.sq_flip1;
    d0 = dy_m; d1 = dx;
    tf0 = flip_sign(py - p.sq_cy, dy_hi);         // sign(d.n0) (p.n0 - cen0) = sign(dy) (py - n0y cen0)
    tf1 = flip_sign(px - p.sq_cx, __double2hiint(dx));
  } else {
    d0 = fma(dx, f.nx[0], dy * f.ny[0]); d1 = fma(dx, f.nx[1], dy * f.ny[1]);
    s0 = __double2hiint(d0); s1 = __double2hiint(d1);
    tf0 = flip_sign(fma(px, f.nx[0], fma(py, f.ny[0], -p.sq_cen0)), s0);
    tf1 = flip_sign(fma(px, f.nx[1], fma(py, f.ny[1], -p.sq_cen1)), s1);
  }
  const double an0 = p.sq_hw0 - tf0, an1 = p.sq_hw1 - tf1;
  // an > 0 by the high word: exact except for 0 < an < 2^-1022
  const bool ok0 = (fabs(d0) >= p.k_eps) & (__double2hiint(an0) > 0), ok1 = (fabs(d1) >= p.k_eps) & (__double2hiint(an1) > 0);
  const int e0 = s0 < 0 ? 2 : 0, e1 = s1 < 0 ? 3 : 1;
  const double l = an0 * fabs(d1), r = an1 * fabs(d0);
  const bool take0 = ok0 & (!ok1 | (l < r) | ((l == r) & (e0 < e1)));
  k = take0 ? e0 : e1;
  const double an = take0 ? an0 : an1, ad = take0 ? d0 : d1;   // |ad| enters the division as an operand modifier
  const bool any = ok0 | ok1;
  u = any ? div_pos_abs(an, ad) : CUDART_INF;
  return any;
}

template <bool SURF, bool UNIFORM, bool REC, bool AXIS>
__device__ __forceinline__ unsigned int sq_ray_loop(const TraceParams& p, const SqBlock& b) {
  const CoarseDev& cf = p.face0;
  // shared-window address of the row histogram, made opaque so that it stays in ONE register: left to itself the compiler
  // rebuilds the window base in front of every atomic (S2UR + UMOV + ULEA + IMAD, 4 issue slots per ray)
  uint32_t hist_s;
  asm volatile("mov.u32 %0, %1;" : "=r"(hist_s) : "r"((uint32_t)__cvta_generic_to_shared(b.hist)));
  unsigned int n_lost = 0;
  // The Philox words of a thread's NEXT ray are computed at the end of the loop body, behind the tally: measured 3 %
  // faster than generating them at the top (11.25 vs 11.53 ms per 1e9 rays) — the integer burst then overlaps the
  // shared-memory atomic and the FP64 tail of the other warps.  (Generating them in the same basic block as the FP64
  // geometry of the current ray, a software pipeline, costs 8 live registers and was slower: 11.62 ms.)
  uint4 w0n, w1n;
  {
    const uint64_t ray_id = (uint64_t)(b.ray0 + (int64_t)threadIdx.x);
    w0n = philox4x32_10_rk(make_uint4((uint32_t)ray_id, (uint32_t)(ray_id >> 32), b.e, b.cw | 0u), p.rk);
    w1n = philox4x32_10_rk(make_uint4((uint32_t)ray_id, (uint32_t)(ray_id >> 32), b.e, b.cw | 1u), p.rk);
  }
  for (uint32_t i = threadIdx.x; i < b.n_rays; i += blockDim.x) {
    const uint4 w0 = w0n, w1 = w1n;
    double px, py, dx, dy, dy_m, R_S;
    int dy_hi;
    emit_ray_folded<SURF>(p, b.s_em, b.sel_thr, w0, w1, px, py, dx, dy, dy_m, dy_hi, R_S);
    if (REC) {
      double* o = p.rec_pts + 4 * (b.rec_base + i);
      o[0] = px; o[1] = py;
    }
    const double neg_log = neg_log_table(R_S, b.s_log);
    int k;
    double u;
    const bool edge = dist_sq<AXIS>(p, px, py, dx, dy, dy_m, dy_hi, u, k);
    double S;
    bool gas, ok = true;
    if (UNIFORM) {
      S = neg_log * b.inv_beta_u;
      gas = S < u;
    } else {
      const int f0 = locate_sq<AXIS>(p, px, py);               // traceRay.jl:87-100
      ok = f0 >= 0;
      const double local_beta = ok ? b.beta_band[f0] : 0.0;
      gas = local_beta * u >= neg_log;
      S = neg_log / local_beta;
    }
    int absorber = -1;
    const bool hit = !gas & edge & (cf.solid[k] != 0);         // an open edge has no neighbour face: the ray is lost
    if (ok & (gas | hit)) {
      const double adv = (gas ? S : u) - p.nudge;
      px = fma(adv, dx, px);
      py = fma(adv, dy, py);
      const int f = locate_sq<AXIS>(p, px, py);
      // gas: Ns + cell; wall: entry 1+k of the cell's absorber-table row = surface index of the fine wall on coarse edge k.
      // Only wall endings load: they touch the boundary cells' rows only, which stay in L1 — loading the
      // gas entry as well made every ray wait on an L1 miss (10 201 rows; long-scoreboard stalls 0.02 -> 1.4 warps per issue).
      if (f >= 0) {
        int sid = p.n_surfaces + f;
        if (!gas) sid = __ldg(p.abs_tab + (unsigned)(f * 5 + 1 + k));
        absorber = sid;
      }
    }
#ifdef RTHX_TALLY_MATCH
    // A/B variant (tools/gpu_evidence_r2.sh builds it as a second library): warp-aggregated tally — lanes that hit the same bin
    // elect one of them to add the group's count.  Measured on cfg3: slower than one red.shared.add.u32 per ray (DESIGN.md section 4).
    {
      const unsigned act = __activemask();
      const unsigned grp = __match_any_sync(act, absorber);
      if (absorber >= 0 && (int)(__ffs((int)grp) - 1) == (int)(threadIdx.x & 31))
        asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(hist_s + 4u * (uint32_t)absorber), "r"((unsigned)__popc(grp)) : "memory");
      if (absorber < 0) ++n_lost;
    }
#else
    if (absorber >= 0) {
      asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(hist_s + 4u * (uint32_t)absorber), "r"(1u) : "memory");
      if (REC) {
        const size_t sl = b.rec_base + i;
        double* o = p.rec_pts + 4 * sl;
        o[2] = px; o[3] = py;
        p.rec_valid[sl] = 1;
      }
    } else {
      ++n_lost;
    }
#endif
    {
      const uint64_t ray_id = (uint64_t)(b.ray0 + (int64_t)(i + blockDim.x));
      w0n = philox4x32_10_rk(make_uint4((uint32_t)ray_id, (uint32_t)(ray_id >> 32), b.e, b.cw | 0u), p.rk);
      w1n = philox4x32_10_rk(make_uint4((uint32_t)ray_id, (uint32_t)(ray_id >> 32), b.e, b.cw | 1u), p.rk);
    }
  }
  return n_lost;
}

// RTHX_MULTI_BOUNCE on the single-quad domain (the analogue of method=:direct's traceSingleRay.jl:7-81 without re-emission): the
// ray is followed through scattering (isotropicScatter2D.jl:1-4) and wall reflection (diffuse: sampleReflectionDirection2D.jl:5-16
// + lambertSample2D; specular: mirror) until it is absorbed; two more Philox calls per event exactly as in trace_exchange_kernel
// <..., MULTI> (call# 2+2n: decision, azimuth, cos(theta), roulette; 3+2n: polar angle, next free path), the same fast arithmetic
// as the first-interaction loop for everything else.
template <bool SURF, bool UNIFORM, bool REC, bool AXIS>
__device__ __forceinline__ unsigned int sq_multi_loop(const TraceParams& p, const SqBlock& b) {
  const CoarseDev& cf = p.face0;
  uint32_t hist_s;
  asm volatile("mov.u32 %0, %1;" : "=r"(hist_s) : "r"((uint32_t)__cvta_generic_to_shared(b.hist)));
  unsigned int n_lost = 0;
  for (uint32_t i = threadIdx.x; i < b.n_rays; i += blockDim.x) {
    const uint64_t ray_id = (uint64_t)(b.ray0 + (int64_t)i);
    const uint32_t c_lo = (uint32_t)ray_id, c_hi = (uint32_t)(ray_id >> 32);
    double px, py, dx, dy, dy_m, R_S;
    int dy_hi;
    {
      const uint4 w0 = philox4x32_10_rk(make_uint4(c_lo, c_hi, b.e, b.cw | 0u), p.rk);
      const uint4 w1 = philox4x32_10_rk(make_uint4(c_lo, c_hi, b.e, b.cw | 1u), p.rk);
      emit_ray_folded<SURF>(p, b.s_em, b.sel_thr, w0, w1, px, py, dx, dy, dy_m, dy_hi, R_S);
    }
    if (REC) {
      double* o = p.rec_pts + 4 * (b.rec_base + i);
      o[0] = px; o[1] = py;
    }
    double neg_log = neg_log_table(R_S, b.s_log);
    int absorber = -1;
#pragma unroll 1
    for (int event = 0;; ++event) {
      // ---- first interaction from (p, d, -log R) ----
      int k;
      double u;
      const bool edge = dist_sq<AXIS>(p, px, py, dx, dy, dy_m, dy_hi, u, k);
      double S;
      bool gas, ok = true;
      if (UNIFORM) {
        S = neg_log * b.inv_beta_u;
        gas = S < u;
      } else {
        const int f0 = locate_sq<AXIS>(p, px, py);
        ok = f0 >= 0;
        const double local_beta = ok ? b.beta_band[f0] : 0.0;
        gas = local_beta * u >= neg_log;
        S = neg_log / local_beta;
      }
      absorber = -1;
      const bool hit = !gas & edge & (cf.solid[k] != 0);
      if (ok & (gas | hit)) {
        const double adv = (gas ? S : u) - p.nudge;
        px = fma(adv, dx, px);
        py = fma(adv, dy, py);
        const int f = locate_sq<AXIS>(p, px, py);
        if (f >= 0) {
          int sid = p.n_surfaces + f;
          if (!gas) sid = __ldg(p.abs_tab + (unsigned)(f * 5 + 1 + k));
          absorber = sid;
        }
      }
      if (absorber < 0) break;                                     // lost
      // ---- absorb, scatter or reflect (traceSingleRay.jl:24-79) ----
      if (event >= 16000) { absorber = -1; break; }                // call# is a 16-bit field
      const uint4 v0 = philox4x32_10_rk(make_uint4(c_lo, c_hi, b.e, b.cw | (uint32_t)(2 + 2 * event)), p.rk);
      const uint4 v1 = philox4x32_10_rk(make_uint4(c_lo, c_hi, b.e, b.cw | (uint32_t)(3 + 2 * event)), p.rk);
      if (event >= 1000 && u32d(v0.w, p.k_u32) > 0.8) { absorber = -1; break; }   // Russian roulette, traceSingleRay.jl:11
      const double dec = u32d(v0.x, p.k_u32);
      if (absorber >= p.n_surfaces) {
        if (!(dec < b.omega_band[absorber - p.n_surfaces])) break;                  // absorbed in the gas
        // isotropicScatter2D.jl:1-4: theta = acos(2R - 1), phi = 2 pi R; with c = R - 1/2: cos = 2c, sin = 2 sqrt(1/4 - c^2)
        const double c = __hiloint2double((int)(0x3FF00000u | (v1.y >> 12)), (int)((v1.y << 20) | (v1.x >> 12))) - p.k_u52c;
        dx = sqrt_pos(fma(-c, c, 0.25)) * cos2pi_centered_x2(u32d_centered(v0.y, p.k_u32c));
        dy = c + c;
      } else {
        if (dec < b.eps_band[absorber]) break;                                      // absorbed by the wall
        const double hnx = cf.nx[k], hny = cf.ny[k];               // outward normal of the coarse edge (= of every fine wall on it)
        if (p.specular) {
          const double dn = dx * hnx + dy * hny;                   // mirror the in-plane components; the axial one is unchanged
          dx = fma(-2.0 * dn, hnx, dx);
          dy = fma(-2.0 * dn, hny, dy);
        } else {
          // diffuse: Lambert about the inward normal n = -hit_n with x-axis (n.y, -n.x)
          const float cosT = __fsqrt_rn(u23(v0.z));
          const float cos2 = __fmul_rn(cosT, cosT);
          const double xdir = sqrt_pos(1.0 - (double)cos2) * cos2pi_centered((double)u23(v0.y) - 0.5);
          const double zdir = (double)cosT;
          const double nxi = -hnx, nyi = -hny;
          const double ndx = nyi * xdir + nxi * zdir;
          dy = -nxi * xdir + nyi * zdir;
          dx = ndx;
        }
      }
      dy_m = dy;
      dy_hi = __double2hiint(dy);
      neg_log = neg_log_table(u52(v1.z, v1.w, p.k_u52), b.s_log);
    }
    if (absorber >= 0) {
      asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(hist_s + 4u * (uint32_t)absorber), "r"(1u) : "memory");
      if (REC) {
        const size_t sl = b.rec_base + i;
        double* o = p.rec_pts + 4 * sl;
        o[2] = px; o[3] = py;
        p.rec_valid[sl] = 1;
      }
    } else {
      ++n_lost;
    }
  }
  return n_lost;
}

template <bool SURF, bool AXIS, bool MULTI>
__device__ __forceinline__ unsigned int sq_dispatch(const TraceParams& p, const SqBlock& b, bool uniform, bool rec) {
  if (MULTI) {
    if (uniform) return rec ? sq_multi_loop<SURF, true, true, AXIS>(p, b) : sq_multi_loop<SURF, true, false, AXIS>(p, b);
    return rec ? sq_multi_loop<SURF, false, true, AXIS>(p, b) : sq_multi_loop<SURF, false, false, AXIS>(p, b);
  }
  if (uniform) return rec ? sq_ray_loop<SURF, true, true, AXIS>(p, b) : sq_ray_loop<SURF, true, false, AXIS>(p, b);
  return rec ? sq_ray_loop<SURF, false, true, AXIS>(p, b) : sq_ray_loop<SURF, false, false, AXIS>(p, b);
}

template <int MINB, bool MULTI>
__global__ void __launch_bounds__(256, MINB) trace_exchange_sq_kernel(const __grid_constant__ TraceParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* s_em = reinterpret_cast<double*>(smem_raw);
  double2* s_log = reinterpret_cast<double2*>(smem_raw + sizeof(double) * EM_DOUBLES);
  uint32_t* hist = reinterpret_cast<uint32_t*>(smem_raw + sizeof(double) * EM_DOUBLES + sizeof(double2) * LOGTAB_N);

  const unsigned bid = blockIdx.x;
  const int chunk = (int)(bid % (unsigned)p.row_chunks);
  const unsigned t1 = bid / (unsigned)p.row_chunks;
  const int bi = (int)(t1 % (unsigned)p.n_bins);
  const int y = p.y_offset + (int)(t1 / (unsigned)p.n_bins);
  const int e = p.emitter_rank + y * p.emitter_world;
  const int band = p.bins[bi];
  const int N = p.N;

  for (int i = threadIdx.x; i < N; i += blockDim.x) hist[i] = 0u;
  for (int i = threadIdx.x; i < LOGTAB_N; i += blockDim.x) s_log[i] = c_logtab[i];
  const int g = p.em_cell[e];
  const int wall = p.em_wall[e];
  const bool is_surface = wall >= 0;
  if (threadIdx.x == 0) stage_emitter_folded(p, g, wall, s_em);

  const int64_t per = (p.rays_per_emitter + p.row_chunks - 1) / p.row_chunks;
  const int64_t r_begin = (int64_t)chunk * per;
  int64_t r_end = r_begin + per;
  if (r_end > p.rays_per_emitter) r_end = p.rays_per_emitter;

  const double ub = p.uniform_beta[band];
  const bool uniform = ub > -0.1;                      // traceRay.jl:4
  const double* beta_band = p.beta + (size_t)band * p.n_cells;
  const double beta_u = beta_band[0];                  // traceRay.jl:6-11: beta of fine_mesh[1][1]
  const int rec_slot = (p.rec_slot != nullptr && band == p.rec_bin) ? p.rec_slot[e] : -1;
  unsigned long long* count_row = p.counts + (p.compact_rows ? ((size_t)bi * p.n_owned + y) : ((size_t)bi * N + e)) * (size_t)N;

  __syncthreads();

  SqBlock b;
  b.s_em = s_em; b.s_log = s_log; b.hist = hist; b.beta_band = beta_band;
  b.inv_beta_u = beta_u > 0.0 ? 1.0 / beta_u : CUDART_INF;
  b.sel_thr = reinterpret_cast<const uint32_t*>(s_em + 15)[0];
  b.omega_band = p.omega + (size_t)band * p.n_cells; b.eps_band = p.eps + (size_t)band * p.n_surfaces;
  b.e = (uint32_t)e; b.cw = ((uint32_t)band << 16);
  b.ray0 = p.ray_id_offset + r_begin;
  b.n_rays = r_end > r_begin ? (uint32_t)(r_end - r_begin) : 0u;
  b.rec_base = rec_slot >= 0 ? (size_t)rec_slot * (size_t)p.rays_per_emitter + (size_t)r_begin : 0;

  unsigned int n_lost;
  const bool rec = rec_slot >= 0;
  if (p.sq_axis) n_lost = is_surface ? sq_dispatch<true, true, MULTI>(p, b, uniform, rec) : sq_dispatch<false, true, MULTI>(p, b, uniform, rec);
  else           n_lost = is_surface ? sq_dispatch<true, false, MULTI>(p, b, uniform, rec) : sq_dispatch<false, false, MULTI>(p, b, uniform, rec);

  for (int off = 16; off > 0; off >>= 1) n_lost += __shfl_down_sync(0xffffffffu, n_lost, off);
  if ((threadIdx.x & 31) == 0 && n_lost) {
    if (p.flush_system) atomicAdd_system(&p.lost[(size_t)bi * N + e], (unsigned long long)n_lost);
    else atomicAdd(&p.lost[(size_t)bi * N + e], (unsigned long long)n_lost);
  }
  __syncthreads();
  if (p.peer_counts != nullptr) { handover_row_hist(p, hist, reinterpret_cast<unsigned int*>(s_em + 15) + 1); return; }
  for (int i = threadIdx.x; i < N; i += blockDim.x) {
    const uint32_t v = hist[i];
    if (v) {
      if (p.flush_system) atomicAdd_system(&count_row[i], (unsigned long long)v);
      else atomicAdd(&count_row[i], (unsigned long long)v);
    }
  }
}

// ------------------------------------------------------------------------------------------------------------
// K1-Q: the fused kernel for multi-face FAST meshes (cfg5: 16 wedges with transparent interfaces and triangle sub-meshes).
// A ray crosses 3-4 coarse faces on average but up to ~10, and in trace_exchange_kernel a warp waits for its longest
// ray: 13.6 of 32 lanes are active on average (ncu), 10.7 in the traversal loop.  Here every warp owns a ray QUEUE in
// shared memory:
//   emission  : each lane emits `depth` rays at full occupancy (Philox + FP64 sampling) and parks their state
//               (p, d, -log R: 40 bytes) in the warp's queue;
//   traversal : one coarse-face step per loop iteration for every lane that holds a ray; lanes whose ray ended take the
//               next unprocessed queue slot — slots are handed out with __ballot_sync + __popc (match / vote, no atomics)
//               — so the warp stays full until its queue runs dry.
// Which lane traces which ray does not matter: tallies are integers keyed by the ray's own Philox counter, so the counts
// stay bit-identical to every other kernel variant, block shape and GPU count.
// ------------------------------------------------------------------------------------------------------------
struct QueueBlock {          // block-uniform state of one (emitter row, band, chunk) in the queue kernel
  const CoarseDev* coarse;   // shared memory
  const double* s_em;
  const double2* s_log;
  uint32_t* hist;
  double* q;                 // this warp's queue, structure of arrays: px | py | dx | dy | S (or -log R), 32*DEPTH doubles each
  const double* beta_band;
  const double* omega_band;  // MULTI_BOUNCE: scattering albedo per cell of the band
  const double* eps_band;    // MULTI_BOUNCE: emissivity per surface of the band
  double inv_beta_u;
  int64_t r_begin, r_end;    // ray range of the block
  size_t rec_row;            // first recorder slot of the emitter row
  uint32_t e, cw, sel_thr;
  int c0, n_warps, warp, lane;
};

// distToSurface2D on a coarse face of the queue kernel (the point is inside the face).
//   parallelogram: slab form about the centre lines as in dist_sq, descriptor fields cen[] / hw[];
//   triangle / general convex quadrilateral: every edge, hit only when moving outward (d.n_i >= eps) with a positive plane distance.
// Sign tests run on the high words, the argmin on cross-multiplied fractions (first index on ties), one division at the end.
template <bool BILIN>
__device__ __forceinline__ bool dist_face(const CoarseDev& f, double px, double py, double dx, double dy, double eps, double& u, int& k) {
  if (f.kind == KIND_AFFINE_QUAD) {
    const double d0 = fma(dx, f.nx[0], dy * f.ny[0]), d1 = fma(dx, f.nx[1], dy * f.ny[1]);
    const int s0 = __double2hiint(d0), s1 = __double2hiint(d1);
    const double tf0 = flip_sign(fma(px, f.nx[0], fma(py, f.ny[0], -f.cen[0])), s0);
    const double tf1 = flip_sign(fma(px, f.nx[1], fma(py, f.ny[1], -f.cen[1])), s1);
    const double an0 = f.hw[0] - tf0, an1 = f.hw[1] - tf1;
    const bool ok0 = (fabs(d0) >= eps) & (__double2hiint(an0) > 0), ok1 = (fabs(d1) >= eps) & (__double2hiint(an1) > 0);
    const int e0 = s0 < 0 ? 2 : 0, e1 = s1 < 0 ? 3 : 1;
    const double l = an0 * fabs(d1), r = an1 * fabs(d0);
    const bool take0 = ok0 & (!ok1 | (l < r) | ((l == r) & (e0 < e1)));
    k = take0 ? e0 : e1;
    const double an = take0 ? an0 : an1, ad = take0 ? d0 : d1;
    const bool any = ok0 | ok1;
    u = any ? div_pos_abs(an, ad) : CUDART_INF;
    return any;
  }
  double bn = 1.0, bd = 0.0;
  int bk = 0;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    if (i == 3 && (!BILIN || f.nv != 4)) break;      // the fourth edge of a general (bilinear-lattice) quadrilateral
    const double nx = f.nx[i], ny = f.ny[i];
    const double den = fma(dx, nx, dy * ny);
    const double num = f.h[i] - fma(px, nx, py * ny);
    const bool better = (den >= eps) & (__double2hiint(num) > 0) & (num * bd < bn * den);
    bn = better ? num : bn;
    bd = better ? den : bd;
    bk = better ? i : bk;
  }
  k = bk;
  const bool any = __double2hiint(bd) > 0;
  u = any ? div_pos(bn, bd) : CUDART_INF;
  return any;
}

// lattice cell n + m Nx of a point in an affine coarse face, or -1 (one unsigned compare per axis, see locate_sq)
// Inverse of the bilinear map P(s,t) = A + s E + t F + s t G of a convex quadrilateral (meshQuad.jl:116-136 divides the unit
// square of (s,t) uniformly): eliminating t gives  a2 s^2 + a1 s + a0 = 0,  a2 = E x G, a1 = E x F - H x G, a0 = -H x F (H = p - A);
// both roots come from the cancellation-free form q = -(a1 + sign(a1) sqrt(disc)) / 2: s = a0 / q or q / a2, the one inside [0,1]
// is the point's (the other lies outside for a convex quadrilateral; a2 = 0, a trapezoid, leaves the first); t by projection of
// H - s E on F + s G.  Verified against the forward map on 3.6e5 random points of random convex quadrilaterals (error < 1e-12).
__device__ __forceinline__ int lattice_cell_bilinear(const CoarseDev& cf, double px, double py) {
  const double hx = px - cf.ax, hy = py - cf.ay;
  const double ex = cf.g1x, ey = cf.g1y, fx = cf.g2x, fy = cf.g2y, gx = cf.cen[0], gy = cf.cen[1];
  const double a2 = ex * gy - ey * gx;
  const double a1 = cf.hw[1] - (hx * gy - hy * gx);
  const double a0 = hy * fx - hx * fy;
  const double disc = fma(a1, a1, -4.0 * a2 * a0);
  if (!(disc >= 0.0)) return -1;
  const double q = -0.5 * (a1 + copysign(sqrt(disc), a1));
  const double sb = a0 / q, sa = q * cf.hw[0];
  const double s = (sb >= -1e-9 && sb <= 1.0 + 1e-9) ? sb : sa;
  const double tx = fma(s, gx, fx), ty = fma(s, gy, fy);
  const double t = (fma(-s, ex, hx) * tx + fma(-s, ey, hy) * ty) / (tx * tx + ty * ty);
  const int n = __double2int_rd(s * (double)cf.Nx), m = __double2int_rd(t * (double)cf.Ny);
  return ((s >= 0.0) & (t >= 0.0) & ((unsigned)n < (unsigned)cf.Nx) & ((unsigned)m < (unsigned)cf.Ny)) ? n + m * cf.Nx : -1;
}

template <bool BILIN>
__device__ __forceinline__ int lattice_cell(const CoarseDev& cf, double px, double py) {
  if (BILIN && cf.kind == KIND_BILINEAR_QUAD) return lattice_cell_bilinear(cf, px, py);
  const double rx = px - cf.ax, ry = py - cf.ay;
  const double s = fma(rx, cf.g1x, ry * cf.g1y), t = fma(rx, cf.g2x, ry * cf.g2y);
  const int n = __double2int_rd(s), m = __double2int_rd(t);
  return (((unsigned)n < (unsigned)cf.Nx) & ((unsigned)m < (unsigned)cf.Ny)) ? n + m * cf.Nx : -1;
}

template <bool SURF, bool UNIFORM, bool REC, int DEPTH, bool BILIN, bool GEN>
__device__ __forceinline__ unsigned int queue_ray_loop(const TraceParams& p, const QueueBlock& b) {
  constexpr int WQ = 32 * DEPTH;                       // queue slots per warp
  const int lane = b.lane;
  double* const q = b.q;                               // field f of slot s at q[f * WQ + s]
  const unsigned lt_mask = (1u << lane) - 1u;
  unsigned int n_lost = 0;
  // Deferred tally (analytic locators, no recorder): the absorber index comes out of a table in global memory (L1 / L2); tallying
  // it on the spot makes the warp wait for the load.  The index is kept in a register instead and tallied in the lane's NEXT step
  // (or behind the loop), a refill and a distToSurface2D later: the load has that long to arrive.
  constexpr bool DEFER = !REC && !GEN;
  constexpr int NO_PEND = INT_MIN;
  int pend_abs = NO_PEND;
#define RTHX_QUEUE_TALLY_PENDING()                     \
  do {                                                 \
    if (DEFER && pend_abs != NO_PEND) {                \
      if (pend_abs >= 0) atomicAdd(&b.hist[pend_abs], 1u); \
      else ++n_lost;                                   \
      pend_abs = NO_PEND;                              \
    }                                                  \
  } while (0)
  // in-flight ray of this lane (lives in registers across queue refills)
  bool active = false;
  double px = 0.0, py = 0.0, dx = 0.0, dy = 0.0, S = 0.0, acc = 0.0;   // S: remaining free path (UNIFORM) or -log R
  int c = b.c0, it = 0;
  uint32_t r_cur = 0;                                  // ray index of the in-flight ray relative to r_begin (recorder slot)
  // the warp's rays: batch j of the block covers [r_begin + j*n_warps*WQ, ...), this warp takes its WQ-slice of every batch
  int64_t rb = b.r_begin + (int64_t)b.warp * WQ;
  const int64_t stride = (int64_t)b.n_warps * WQ;
  while (true) {
    // ---- stage 1: emission at full occupancy into the warp's queue ----------------------------------------------------
    const int n_valid = rb < b.r_end ? (int)min((int64_t)WQ, b.r_end - rb) : 0;
#pragma unroll 1
    for (int s = lane; s < n_valid; s += 32) {
      const uint64_t ray_id = (uint64_t)(p.ray_id_offset + rb + s);
      const uint32_t c_lo = (uint32_t)ray_id, c_hi = (uint32_t)(ray_id >> 32);
      const uint4 w0 = philox4x32_10_rk(make_uint4(c_lo, c_hi, b.e, b.cw | 0u), p.rk);
      const uint4 w1 = philox4x32_10_rk(make_uint4(c_lo, c_hi, b.e, b.cw | 1u), p.rk);
      double ex, ey, fx, fy, fy_m, R_S;
      int fy_hi;
      emit_ray_folded<SURF>(p, b.s_em, b.sel_thr, w0, w1, ex, ey, fx, fy, fy_m, fy_hi, R_S);
      if (REC) {
        double* o = p.rec_pts + 4 * (b.rec_row + (size_t)(rb + s));
        o[0] = ex; o[1] = ey;
      }
      const double nl = neg_log_table(R_S, b.s_log);
      q[s] = ex; q[WQ + s] = ey; q[2 * WQ + s] = fx; q[3 * WQ + s] = fy; q[4 * WQ + s] = UNIFORM ? nl * b.inv_beta_u : nl;
    }
    __syncwarp();
    const bool last_batch = rb + stride >= b.r_end;    // nothing left to emit after this queue
    const uint32_t rb_rel = (uint32_t)(rb - b.r_begin);
    // ---- stage 2: traversal; idle lanes take queue slots by warp vote --------------------------------------------------
    int next = 0;
    while (true) {
      // refill: every lane without a ray takes the next unprocessed slot
      const unsigned need = __ballot_sync(0xffffffffu, !active);
      const int idx = next + __popc(need & lt_mask);
      if (!active & (idx < n_valid)) {
        px = q[idx]; py = q[WQ + idx]; dx = q[2 * WQ + idx]; dy = q[3 * WQ + idx]; S = q[4 * WQ + idx];
        acc = 0.0; c = b.c0; it = 0; r_cur = rb_rel + (uint32_t)idx;
        active = true;
      }
      next += __popc(need);
      const unsigned busy = __ballot_sync(0xffffffffu, active);
      if (busy == 0u) break;                                           // queue dry and nothing in flight
      if (next >= n_valid && !last_batch && __popc(busy) <= p.queue_refill) break; // queue dry: emit the next batch at full occupancy,
                                                                       // the in-flight rays stay in their lanes
      // one step = distToSurface2D on the current coarse face + ONE advance shared by the three outcomes (gas event, solid
      // wall, crossing: only the advance length differs); the only divergent region is "this ray ended"
      if (active) {
        const CoarseDev& cf = b.coarse[c];
        // GEN (a general variant of its own, so that meshes of analytic faces keep their registers): faces without an analytic
        // locator, and every face under RTHX_LOCATOR_GENERIC, are located by bucket grid + crossing number
        const bool gen = GEN && (p.force_generic != 0 || cf.kind == KIND_GENERIC);
        int k;
        double u;
        const bool edge = dist_face<BILIN>(cf, px, py, dx, dy, p.k_eps, u, k);  // an edge lies ahead
        RTHX_QUEUE_TALLY_PENDING();                                            // the ending of this lane's previous ray
        bool gas, ok = true;
        double tau_b = 0.0, Sg;
        if (UNIFORM) {
          gas = S < u;
          Sg = S;
        } else {
          int f0;                                                              // traceRay.jl:87-100
          if (GEN && gen) {
            f0 = find_face_generic(p, 1 + c, px, py);
          } else {
            const int l0 = lattice_cell<BILIN>(cf, px, py);
            f0 = l0 < 0 ? -1 : (cf.kind == KIND_AFFINE_TRI ? __ldg(p.lattice + cf.lat_off + l0) : l0);
          }
          ok = f0 >= 0;
          const double local_beta = ok ? b.beta_band[cf.fine_off + f0] : 0.0;
          tau_b = local_beta * u;
          gas = acc + tau_b >= S;
          Sg = (S - acc) / local_beta;
        }
        const bool solid = cf.solid[k] != 0;
        const int nc = cf.nbr[k];
        // BILIN (the general variant) also serves interfaces without a unique neighbour face — T-junctions, open edges — by the
        // reference's own coarse point location after the advance (traceRay.jl:56-65)
        const bool cross = ok & !gas & edge & !solid & (BILIN | (nc >= 0)) & (it < 9999);
        const bool tallied = ok & (gas | (edge & solid));               // ends in an element (unless the location fails)
        // traceRay.jl:33,44,56: gas S - nudge, solid wall u - nudge, crossing u + nudge
        const double adv = gas ? Sg - p.nudge : (solid ? u - p.nudge : u + p.nudge);
        if (cross | tallied) {
          px = fma(adv, dx, px);
          py = fma(adv, dy, py);
        }
        // GEN: ONE call of the generic locator per iteration serves both kinds of lane — the coarse face behind a crossing (set 0)
        // and the fine cell a ray ends in (set 1 + c).  With a call in each branch the warp ran the locator twice per iteration at
        // ~12 of 32 lanes (ncu: 2810 warp instructions per 32 rays on cfg5).
        const bool loc_cross = GEN && cross && (p.force_generic != 0 || nc < 0);   // RTHX_LOCATOR_GENERIC: the reference's search after every crossing
        const bool loc_end = GEN && gen && !cross && tallied;
        int loc = -1;
        if (GEN && (loc_cross | loc_end)) loc = find_face_generic(p, loc_cross ? 0 : 1 + c, px, py);
        // a ray that ends: absorber index of (lattice cell, gas | wall on coarse edge k) in ONE table load shared by both endings
        // (rthx_api.cu builds the table from the lattice -> fine map, the fine cells' vertex counts and cell_surf_id)
#define RTHX_QUEUE_FINISH()                                                                                         \
  do {                                                                                                              \
    active = false;                                                                                                 \
    int absorber = -1;                                                                                              \
    if (tallied) {                                                                                                  \
      if (GEN && gen) {                                                                                             \
        const int f = loc;                                                                                          \
        if (f >= 0) {                                                                                               \
          if (gas) absorber = p.n_surfaces + cf.fine_off + f;                                                       \
          else wall_of_rec(p.face_rec + 12 * (size_t)(cf.fine_off + f), px, py, dx, dy, absorber); /* traceRay.jl:51 */ \
        }                                                                                                           \
      } else {                                                                                                      \
        const int l = lattice_cell<BILIN>(cf, px, py);                                                              \
        if (l >= 0) absorber = __ldg(p.abs_tab + (size_t)(cf.abs_off + l) * 5 + (gas ? 0 : 1 + k));                 \
      }                                                                                                             \
    }                                                                                                               \
    if (DEFER) {                                                                                                    \
      pend_abs = absorber;                       /* tallied by RTHX_QUEUE_TALLY_PENDING in the lane's next step */     \
    } else if (absorber >= 0) {                                                                                     \
      atomicAdd(&b.hist[absorber], 1u);                                                                             \
      if (REC) {                                                                                                    \
        const size_t sl = b.rec_row + (size_t)(b.r_begin + (int64_t)r_cur);                                         \
        double* o = p.rec_pts + 4 * sl;                                                                             \
        o[2] = px; o[3] = py;                                                                                       \
        p.rec_valid[sl] = 1;                                                                                        \
      }                                                                                                             \
    } else {                                                                                                        \
      ++n_lost;                                                                                                     \
    }                                                                                                               \
  } while (0)
        if (!BILIN) {
          if (cross) {
            if (UNIFORM) S -= u; else acc += tau_b;
            c = nc;
            ++it;
          } else {
            RTHX_QUEUE_FINISH();
          }
        } else {
          bool ended = !cross;
          if (cross) {
            if (UNIFORM) S -= u; else acc += tau_b;
            int nn;
            if (GEN) {
              nn = loc_cross ? loc : nc;
            } else {
              nn = nc;
              if (nn < 0) nn = find_face_generic(p, 0, px, py);
            }
            if (nn >= 0) { c = nn; ++it; }
            else ended = true;                                           // left the domain: lost, like the reference's `nothing`
          }
          if (ended) RTHX_QUEUE_FINISH();                                // (a failed crossing has tallied == false: counted as lost)
        }
#undef RTHX_QUEUE_FINISH
      }
    }
    __syncwarp();
    if (last_batch) break;                             // the inner loop only leaves the last batch with nothing in flight
    rb += stride;
  }
  RTHX_QUEUE_TALLY_PENDING();                          // lanes that took no further ray
#undef RTHX_QUEUE_TALLY_PENDING
  return n_lost;
}

template <bool SURF, int DEPTH, bool BILIN, bool GEN>
__device__ __forceinline__ unsigned int queue_dispatch(const TraceParams& p, const QueueBlock& b, bool uniform, bool rec) {
  if (uniform) return rec ? queue_ray_loop<SURF, true, true, DEPTH, BILIN, GEN>(p, b) : queue_ray_loop<SURF, true, false, DEPTH, BILIN, GEN>(p, b);
  return rec ? queue_ray_loop<SURF, false, true, DEPTH, BILIN, GEN>(p, b) : queue_ray_loop<SURF, false, false, DEPTH, BILIN, GEN>(p, b);
}

// ------------------------------------------------------------------------------------------------------------
// K1-QM: RTHX_MULTI_BOUNCE[_SPECULAR] on the ray queue — the analogue of method=:direct's traceSingleRay.jl:24-79 without
// re-emission, in two phases per warp so that every phase runs on full warps:
//   produce : (a) rays that survived an interaction ("pending": interaction point, incoming direction, the Philox words of the
//             event) get their new direction — isotropic scattering (isotropicScatter2D.jl:1-4), diffuse reflection about the
//             inward wall normal (sampleReflectionDirection2D.jl:5-16 + lambertSample2D) or a mirror reflection — and their next
//             free path, one lane per ray; (b) the rest of the queue is topped up with freshly emitted rays;
//   consume : as in queue_ray_loop, one coarse-face step per iteration for every lane that holds a ray; a ray that interacts
//             draws its fate (one Philox call: absorbed / continues / Russian roulette, :11) right there, is tallied if absorbed
//             and otherwise parked as a pending entry in a slot of the queue that was already consumed; the lane refills.
// In the lock-step loop (sq_multi_loop) a warp waits for its longest event chain: 15.5 of 32 lanes on cfg3 with omega = 0.5.
// Which lane continues which ray is irrelevant for the result: every draw is keyed by (ray id, emitter, band, call#), call#
// 2+2n / 3+2n for event n exactly as in trace_exchange_kernel<..., MULTI>, so the tallies stay bit-identical to it.
// Slot layout (structure of arrays over the WQ slots of a warp): px | py | dx | dy | S as doubles, rid | meta as u32;
//   meta = event | coarse face << 14 | (pending only) edge << 23 | gas << 25; a pending entry keeps (v0.y, v0.z) in the S slot.
// ------------------------------------------------------------------------------------------------------------
//   SQK: 0 = any mesh with analytic locators (coarse descriptors in shared memory); 1 / 2 = the whole domain is ONE parallelogram
//        (axis-aligned / general): the consume step is the SQ kernel's — face constants from the kernel-parameter bank, slab distance,
//        folded lattice inverse, no crossings — and there is no coarse index to carry.
template <bool SURF, bool UNIFORM, bool REC, int DEPTH, bool BILIN, int SQK>
__device__ __forceinline__ unsigned int queue_multi_loop(const TraceParams& p, const QueueBlock& b) {
  constexpr int WQ = 32 * DEPTH;
  const int lane = b.lane;
  double* const q = b.q;                               // field f of slot s at q[f * WQ + s]
  uint32_t* const qi = reinterpret_cast<uint32_t*>(q + 5 * WQ);   // rid at qi[s], meta at qi[WQ + s]
  const unsigned lt_mask = (1u << lane) - 1u;
  unsigned int n_lost = 0;
  // in-flight ray of this lane
  bool active = false;
  double px = 0.0, py = 0.0, dx = 0.0, dy = 0.0, S = 0.0, acc = 0.0;
  int c = b.c0, it = 0, event = 0;
  uint32_t r_cur = 0;
  // this warp's contiguous share of the block's rays (indices relative to r_begin)
  const int64_t n_block = b.r_end - b.r_begin;
  const int64_t per_warp = (n_block + b.n_warps - 1) / b.n_warps;
  int64_t r_next = min(n_block, (int64_t)b.warp * per_warp);
  const int64_t r_stop = min(n_block, r_next + per_warp);
  int n_pend = 0;                                      // parked survivors, slots [0, n_pend); they persist across phases
  while (true) {
    // ---- produce ---------------------------------------------------------------------------------------------------------
    // Both halves run on FULL warps: survivors are converted in groups of 32 (the rest stays parked for a later phase) and fresh
    // rays are emitted in groups of 32, except when the warp's rays run out (then everything parked is converted).
    const int64_t remaining = r_stop - r_next;
    int n_conv = remaining > 0 ? (n_pend & ~31) : n_pend;
    int n_fresh = (int)min((int64_t)(WQ - n_pend), remaining);
    if ((int64_t)n_fresh < remaining) n_fresh &= ~31;
    if (n_conv == 0 && n_fresh == 0) { n_conv = n_pend; n_fresh = (int)min((int64_t)(WQ - n_pend), remaining); }   // progress (shallow queues)
    const int keep = n_pend - n_conv;                  // slots [0, keep) stay parked; [keep, n_pend) become ready in place
    // (a) pending -> ready, in place, one lane per ray
#pragma unroll 1
    for (int s = keep + lane; s < n_pend; s += 32) {
      const uint32_t rid = qi[s], meta = qi[WQ + s];
      const int ev = (int)(meta & 0x3FFFu), cc = (int)((meta >> 14) & 0x1FFu), k = (int)((meta >> 23) & 3u);
      const bool gas = (meta >> 25) & 1u;
      const uint2 v0yz = *reinterpret_cast<const uint2*>(&q[4 * WQ + s]);       // (v0.y, v0.z) of the event's first call
      const uint64_t ray_id = (uint64_t)(p.ray_id_offset + b.r_begin + (int64_t)rid);
      const uint4 v1 = philox4x32_10_rk(make_uint4((uint32_t)ray_id, (uint32_t)(ray_id >> 32), b.e, b.cw | (uint32_t)(3 + 2 * ev)), p.rk);
      double ndx, ndy;
      if (gas) {
        // theta = acos(2R - 1), phi = 2 pi R; with c = R - 1/2: cos = 2c, sin = 2 sqrt(1/4 - c^2)
        const double ch = __hiloint2double((int)(0x3FF00000u | (v1.y >> 12)), (int)((v1.y << 20) | (v1.x >> 12))) - p.k_u52c;
        ndx = sqrt_pos(fma(-ch, ch, 0.25)) * cos2pi_centered_x2(u32d_centered(v0yz.x, p.k_u32c));
        ndy = ch + ch;
      } else {
        const CoarseDev& cf = SQK ? p.face0 : b.coarse[cc];
        const double hnx = cf.nx[k], hny = cf.ny[k];                 // outward normal of the coarse edge (= of every fine wall on it)
        if (p.specular) {
          const double idx_ = q[2 * WQ + s], idy_ = q[3 * WQ + s];   // incoming direction: mirror the in-plane components
          const double dn = idx_ * hnx + idy_ * hny;
          ndx = fma(-2.0 * dn, hnx, idx_);
          ndy = fma(-2.0 * dn, hny, idy_);
        } else {
          // Lambert about the inward normal n = -hit_n with x-axis (n.y, -n.x)
          const float cosT = __fsqrt_rn(u23(v0yz.y));
          const float cos2 = __fmul_rn(cosT, cosT);
          const double xdir = sqrt_pos(1.0 - (double)cos2) * cos2pi_centered((double)u23(v0yz.x) - 0.5);
          const double zdir = (double)cosT;
          const double nxi = -hnx, nyi = -hny;
          ndx = nyi * xdir + nxi * zdir;
          ndy = -nxi * xdir + nyi * zdir;
        }
      }
      const double nl = neg_log_table(u52(v1.z, v1.w, p.k_u52), b.s_log);
      q[2 * WQ + s] = ndx; q[3 * WQ + s] = ndy; q[4 * WQ + s] = UNIFORM ? nl * b.inv_beta_u : nl;
      qi[WQ + s] = (uint32_t)(ev + 1) | ((uint32_t)cc << 14);
    }
    // (b) fresh rays behind them
#pragma unroll 1
    for (int s = lane; s < n_fresh; s += 32) {
      const uint32_t rid = (uint32_t)(r_next + s);
      const uint64_t ray_id = (uint64_t)(p.ray_id_offset + b.r_begin + (int64_t)rid);
      const uint32_t c_lo = (uint32_t)ray_id, c_hi = (uint32_t)(ray_id >> 32);
      const uint4 w0 = philox4x32_10_rk(make_uint4(c_lo, c_hi, b.e, b.cw | 0u), p.rk);
      const uint4 w1 = philox4x32_10_rk(make_uint4(c_lo, c_hi, b.e, b.cw | 1u), p.rk);
      double ex, ey, fx, fy, fy_m, R_S;
      int fy_hi;
      emit_ray_folded<SURF>(p, b.s_em, b.sel_thr, w0, w1, ex, ey, fx, fy, fy_m, fy_hi, R_S);
      if (REC) {
        double* o = p.rec_pts + 4 * (b.rec_row + (size_t)(b.r_begin + (int64_t)rid));
        o[0] = ex; o[1] = ey;
      }
      const double nl = neg_log_table(R_S, b.s_log);
      const int t = n_pend + s;
      q[t] = ex; q[WQ + t] = ey; q[2 * WQ + t] = fx; q[3 * WQ + t] = fy; q[4 * WQ + t] = UNIFORM ? nl * b.inv_beta_u : nl;
      qi[t] = rid; qi[WQ + t] = (uint32_t)b.c0 << 14;
    }
    const int n_valid = n_pend + n_fresh;              // ready rays: slots [keep, n_valid)
    r_next += n_fresh;
    n_pend = keep;
    __syncwarp();
    if (n_valid == keep && __ballot_sync(0xffffffffu, active) == 0u) break;   // nothing ready, nothing in flight (then nothing is parked either)
    const bool more_fresh = r_next < r_stop;
    // ---- consume ----------------------------------------------------------------------------------------------------------
    int next = keep;
    while (true) {
      // refill: every lane without a ray takes the next unprocessed slot
      const unsigned need = __ballot_sync(0xffffffffu, !active);
      const int idx = next + __popc(need & lt_mask);
      if (!active & (idx < n_valid)) {
        px = q[idx]; py = q[WQ + idx]; dx = q[2 * WQ + idx]; dy = q[3 * WQ + idx]; S = q[4 * WQ + idx];
        r_cur = qi[idx];
        const uint32_t meta = qi[WQ + idx];
        event = (int)(meta & 0x3FFFu); c = (int)(meta >> 14);
        acc = 0.0; it = 0;
        active = true;
      }
      next = min(next + __popc(need), n_valid);
      const unsigned busy = __ballot_sync(0xffffffffu, active);
      if (busy == 0u) break;                                           // queue dry and nothing in flight
      // queue dry while more rays can be produced (fresh ones or parked survivors): go and produce at full occupancy once few
      // lanes still hold a ray; those rays stay in their lanes
      if (next >= n_valid && (more_fresh | (n_pend > 0)) && __popc(busy) <= p.queue_refill) break;
      bool park = false;                                               // this lane's ray survived an interaction
      uint32_t park_meta = 0u, park_y = 0u, park_z = 0u;
      if (active) {
        int k;
        bool gas, ended = true;
        int absorber = -1;
        if constexpr (SQK != 0) {
          // single parallelogram: one distToSurface2D, one decision, one fine-cell location (traceRay.jl:27-52), as in sq_ray_loop
          constexpr bool AXIS = SQK == 1;
          const CoarseDev& cf = p.face0;
          double u;
          const bool edge = dist_sq<AXIS>(p, px, py, dx, dy, dy, __double2hiint(dy), u, k);
          bool ok = true;
          double Sg;
          if (UNIFORM) {
            gas = S < u;
            Sg = S;
          } else {
            const int f0 = locate_sq<AXIS>(p, px, py);                           // traceRay.jl:87-100
            ok = f0 >= 0;
            const double local_beta = ok ? b.beta_band[f0] : 0.0;
            gas = local_beta * u >= S;
            Sg = S / local_beta;
          }
          const bool hit = !gas & edge & (cf.solid[k] != 0);                     // an open edge has no neighbour face: the ray is lost
          if (ok & (gas | hit)) {
            const double adv = (gas ? Sg : u) - p.nudge;
            px = fma(adv, dx, px);
            py = fma(adv, dy, py);
            const int f = locate_sq<AXIS>(p, px, py);
            if (f >= 0) absorber = gas ? p.n_surfaces + f : __ldg(p.abs_tab + (unsigned)(f * 5 + 1 + k));
          }
        } else {
          const CoarseDev& cf = b.coarse[c];
          double u;
          const bool edge = dist_face<BILIN>(cf, px, py, dx, dy, p.k_eps, u, k);
          bool ok = true;
          double tau_b = 0.0, Sg;
          if (UNIFORM) {
            gas = S < u;
            Sg = S;
          } else {
            const int l0 = lattice_cell<BILIN>(cf, px, py);                      // traceRay.jl:87-100
            const int f0 = l0 < 0 ? -1 : (cf.kind == KIND_AFFINE_TRI ? __ldg(p.lattice + cf.lat_off + l0) : l0);
            ok = f0 >= 0;
            const double local_beta = ok ? b.beta_band[cf.fine_off + f0] : 0.0;
            tau_b = local_beta * u;
            gas = acc + tau_b >= S;
            Sg = (S - acc) / local_beta;
          }
          const bool solid = cf.solid[k] != 0;
          const int nc = cf.nbr[k];
          const bool cross = ok & !gas & edge & !solid & (BILIN | (nc >= 0)) & (it < 9999);
          const bool tallied = ok & (gas | (edge & solid));
          const double adv = gas ? Sg - p.nudge : (solid ? u - p.nudge : u + p.nudge);
          if (cross | tallied) {
            px = fma(adv, dx, px);
            py = fma(adv, dy, py);
          }
          ended = !cross;
          if (cross) {
            if (UNIFORM) S -= u; else acc += tau_b;
            int nn = nc;
            if (BILIN) { if (nn < 0) nn = find_face_generic(p, 0, px, py); }
            if (nn >= 0) { c = nn; ++it; }
            else ended = true;                                           // left the domain: lost, like the reference's `nothing`
          }
          if (ended & tallied) {
            const int l = lattice_cell<BILIN>(cf, px, py);
            if (l >= 0) absorber = (gas & (cf.kind != KIND_AFFINE_TRI)) ? p.n_surfaces + cf.fine_off + l
                                                                        : __ldg(p.abs_tab + (size_t)(cf.abs_off + l) * 5 + (gas ? 0 : 1 + k));
          }
        }
        if (ended) {
          if (absorber >= 0) {
            // absorb, or live on (traceSingleRay.jl:24-79): v0.x decision, v0.w roulette; v0.y / v0.z feed the new direction
            if (event >= 16000) {                                      // call# is a 16-bit field
              absorber = -1;
            } else {
              // albedo of the cell / emissivity of the wall.  The per-cell albedo array (80 KB for cfg3) lives in L2: where a band has
              // ONE albedo (p.band_u, staged in the emitter block) the load is skipped — ptxas sinks it behind the ten Philox
              // rounds whatever the source order, and the event then waits for L2 (long_scoreboard 1.6 cycles per issue)
              const bool in_gas = absorber >= p.n_surfaces;
              double lim = b.s_em[in_gas ? 13 : 12];                   // the band's albedo / emissivity where all cells / walls share one (or -1)
              if (lim < 0.0) lim = __ldg(in_gas ? b.omega_band + (absorber - p.n_surfaces) : b.eps_band + absorber);
              const uint64_t ray_id = (uint64_t)(p.ray_id_offset + b.r_begin + (int64_t)r_cur);
              const uint4 v0 = philox4x32_10_rk(make_uint4((uint32_t)ray_id, (uint32_t)(ray_id >> 32), b.e, b.cw | (uint32_t)(2 + 2 * event)), p.rk);
              if (event >= 1000 && u32d(v0.w, p.k_u32) > 0.8) {        // Russian roulette, traceSingleRay.jl:11
                absorber = -1;
              } else {
                const double dec = u32d(v0.x, p.k_u32);
                park = in_gas ? (dec < lim) : !(dec < lim);
                park_meta = (uint32_t)event | ((uint32_t)c << 14) | ((uint32_t)k << 23) | (gas ? (1u << 25) : 0u);
                park_y = v0.y; park_z = v0.z;
              }
            }
          }
          if (!park) {
            active = false;
            if (absorber >= 0) {
              atomicAdd(&b.hist[absorber], 1u);
              if (REC) {
                const size_t sl = b.rec_row + (size_t)(b.r_begin + (int64_t)r_cur);
                double* o = p.rec_pts + 4 * sl;
                o[2] = px; o[3] = py;
                p.rec_valid[sl] = 1;
              }
            } else {
              ++n_lost;
            }
          }
        }
      }
      // park the survivors in consumed slots: [0, next) while the queue still holds rays, the whole buffer once it is dry
      const unsigned pm = __ballot_sync(0xffffffffu, park);
      if (pm) {
        __syncwarp();                                                  // this iteration's refill loads are done before slots are overwritten
        const int cap = next >= n_valid ? WQ : next;
        const int slot = n_pend + __popc(pm & lt_mask);
        if (park) {
          if (slot < cap) {
            q[slot] = px; q[WQ + slot] = py; q[2 * WQ + slot] = dx; q[3 * WQ + slot] = dy;
            *reinterpret_cast<uint2*>(&q[4 * WQ + slot]) = make_uint2(park_y, park_z);
            qi[slot] = r_cur; qi[WQ + slot] = park_meta;
            active = false;
          } else {
            // no free slot (only rays carried over a produce phase can outnumber the consumed slots): continue in the lane
            const int k = (int)((park_meta >> 23) & 3u);
            const uint64_t ray_id = (uint64_t)(p.ray_id_offset + b.r_begin + (int64_t)r_cur);
            const uint4 v1 = philox4x32_10_rk(make_uint4((uint32_t)ray_id, (uint32_t)(ray_id >> 32), b.e, b.cw | (uint32_t)(3 + 2 * event)), p.rk);
            if ((park_meta >> 25) & 1u) {
              const double ch = __hiloint2double((int)(0x3FF00000u | (v1.y >> 12)), (int)((v1.y << 20) | (v1.x >> 12))) - p.k_u52c;
              dx = sqrt_pos(fma(-ch, ch, 0.25)) * cos2pi_centered_x2(u32d_centered(park_y, p.k_u32c));
              dy = ch + ch;
            } else {
              const CoarseDev& cf = SQK ? p.face0 : b.coarse[c];
              const double hnx = cf.nx[k], hny = cf.ny[k];
              if (p.specular) {
                const double dn = dx * hnx + dy * hny;
                dx = fma(-2.0 * dn, hnx, dx);
                dy = fma(-2.0 * dn, hny, dy);
              } else {
                const float cosT = __fsqrt_rn(u23(park_z));
                const float cos2 = __fmul_rn(cosT, cosT);
                const double xdir = sqrt_pos(1.0 - (double)cos2) * cos2pi_centered((double)u23(park_y) - 0.5);
                const double zdir = (double)cosT;
                const double nxi = -hnx, nyi = -hny;
                dx = nyi * xdir + nxi * zdir;
                dy = -nxi * xdir + nyi * zdir;
              }
            }
            const double nl = neg_log_table(u52(v1.z, v1.w, p.k_u52), b.s_log);
            S = UNIFORM ? nl * b.inv_beta_u : nl;
            acc = 0.0; it = 0; ++event;
          }
        }
        n_pend = min(cap, n_pend + __popc(pm));
      }
    }
    __syncwarp();
  }
  return n_lost;
}

template <bool SURF, int DEPTH, bool BILIN, int SQK>
__device__ __forceinline__ unsigned int queue_multi_dispatch(const TraceParams& p, const QueueBlock& b, bool uniform, bool rec) {
  if (uniform) return rec ? queue_multi_loop<SURF, true, true, DEPTH, BILIN, SQK>(p, b) : queue_multi_loop<SURF, true, false, DEPTH, BILIN, SQK>(p, b);
  return rec ? queue_multi_loop<SURF, false, true, DEPTH, BILIN, SQK>(p, b) : queue_multi_loop<SURF, false, false, DEPTH, BILIN, SQK>(p, b);
}

// BILIN: the mesh has general convex quadrilateral faces (bilinear lattices); compiled separately so that meshes of parallelograms
// and triangles keep the shorter traversal loop
template <int MINB, int DEPTH, bool BILIN, bool MULTI, bool GEN = false>
__global__ void __launch_bounds__(256, MINB) trace_exchange_queue_kernel(const __grid_constant__ TraceParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const size_t coarse_bytes = sizeof(CoarseDev) * (size_t)p.n_coarse;
  double* s_em = reinterpret_cast<double*>(smem_raw + coarse_bytes);
  double2* s_log = reinterpret_cast<double2*>(smem_raw + coarse_bytes + sizeof(double) * EM_DOUBLES);
  uint32_t* hist = reinterpret_cast<uint32_t*>(smem_raw + coarse_bytes + sizeof(double) * EM_DOUBLES + sizeof(double2) * LOGTAB_N);
  const int N = p.N;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
  constexpr int WQ = 32 * DEPTH;
  double* queue = reinterpret_cast<double*>(smem_raw + ((coarse_bytes + sizeof(double) * EM_DOUBLES + sizeof(double2) * LOGTAB_N + sizeof(uint32_t) * (size_t)N + 15) & ~size_t(15)));

  const unsigned bid = blockIdx.x;
  const int chunk = (int)(bid % (unsigned)p.row_chunks);
  const unsigned t1 = bid / (unsigned)p.row_chunks;
  const int bi = (int)(t1 % (unsigned)p.n_bins);
  const int y = p.y_offset + (int)(t1 / (unsigned)p.n_bins);
  const int e = p.emitter_rank + y * p.emitter_world;
  const int band = p.bins[bi];

  {
    const int nw = (int)(coarse_bytes / 8);
    const double* src = reinterpret_cast<const double*>(p.coarse);
    double* dst = reinterpret_cast<double*>(smem_raw);
    for (int i = threadIdx.x; i < nw; i += blockDim.x) dst[i] = src[i];
  }
  for (int i = threadIdx.x; i < N; i += blockDim.x) hist[i] = 0u;
  for (int i = threadIdx.x; i < LOGTAB_N; i += blockDim.x) s_log[i] = c_logtab[i];

  const int g = p.em_cell[e];
  const int wall = p.em_wall[e];
  const bool is_surface = wall >= 0;
  if (threadIdx.x == 0) { stage_emitter_folded(p, g, wall, s_em); if (MULTI) { s_em[12] = p.band_u[2 * band + 1]; s_em[13] = p.band_u[2 * band]; } }   // [12], [13]: free slots of the emitter block

  const int64_t per = (p.rays_per_emitter + p.row_chunks - 1) / p.row_chunks;
  const int64_t r_begin = (int64_t)chunk * per;
  int64_t r_end = r_begin + per;
  if (r_end > p.rays_per_emitter) r_end = p.rays_per_emitter;

  const double ub = p.uniform_beta[band];
  const bool uniform = ub > -0.1;                      // traceRay.jl:4
  const double* beta_band = p.beta + (size_t)band * p.n_cells;
  const double beta_u = beta_band[0];                  // traceRay.jl:6-11: beta of fine_mesh[1][1]
  const int rec_slot = (p.rec_slot != nullptr && band == p.rec_bin) ? p.rec_slot[e] : -1;
  unsigned long long* count_row = p.counts + (p.compact_rows ? ((size_t)bi * p.n_owned + y) : ((size_t)bi * N + e)) * (size_t)N;

  __syncthreads();

  QueueBlock b;
  b.coarse = reinterpret_cast<const CoarseDev*>(smem_raw);
  b.s_em = s_em; b.s_log = s_log; b.hist = hist;
  b.q = queue + (size_t)warp * (MULTI ? 6 : 5) * WQ;          // MULTI: + rid / meta words per slot
  b.beta_band = beta_band;
  b.omega_band = p.omega + (size_t)band * p.n_cells; b.eps_band = p.eps + (size_t)band * p.n_surfaces;
  b.inv_beta_u = beta_u > 0.0 ? 1.0 / beta_u : CUDART_INF;
  b.r_begin = r_begin; b.r_end = r_end;
  b.rec_row = rec_slot >= 0 ? (size_t)rec_slot * (size_t)p.rays_per_emitter : 0;
  b.e = (uint32_t)e; b.cw = ((uint32_t)band << 16);
  b.sel_thr = reinterpret_cast<const uint32_t*>(s_em + 15)[0];
  b.c0 = p.em_coarse[e]; b.n_warps = n_warps; b.warp = warp; b.lane = lane;

  unsigned int n_lost0;
  if (MULTI) {
    // a single parallelogram (p.queue_sq: 1 axis-aligned, 2 general) takes the SQ form of the step; BILIN instances never do
    if (!BILIN && p.queue_sq == 1) n_lost0 = is_surface ? queue_multi_dispatch<true, DEPTH, false, 1>(p, b, uniform, rec_slot >= 0) : queue_multi_dispatch<false, DEPTH, false, 1>(p, b, uniform, rec_slot >= 0);
    else if (!BILIN && p.queue_sq == 2) n_lost0 = is_surface ? queue_multi_dispatch<true, DEPTH, false, 2>(p, b, uniform, rec_slot >= 0) : queue_multi_dispatch<false, DEPTH, false, 2>(p, b, uniform, rec_slot >= 0);
    else n_lost0 = is_surface ? queue_multi_dispatch<true, DEPTH, BILIN, 0>(p, b, uniform, rec_slot >= 0) : queue_multi_dispatch<false, DEPTH, BILIN, 0>(p, b, uniform, rec_slot >= 0);
  }
  else n_lost0 = is_surface ? queue_dispatch<true, DEPTH, BILIN, GEN>(p, b, uniform, rec_slot >= 0) : queue_dispatch<false, DEPTH, BILIN, GEN>(p, b, uniform, rec_slot >= 0);
  unsigned int n_lost = n_lost0;

  // ---- flush --------------------------------------------------------------------------------------------------
  for (int off = 16; off > 0; off >>= 1) n_lost += __shfl_down_sync(0xffffffffu, n_lost, off);
  if (lane == 0 && n_lost) {
    if (p.flush_system) atomicAdd_system(&p.lost[(size_t)bi * N + e], (unsigned long long)n_lost);
    else atomicAdd(&p.lost[(size_t)bi * N + e], (unsigned long long)n_lost);
  }
  __syncthreads();
  if (p.peer_counts != nullptr) { handover_row_hist(p, hist, reinterpret_cast<unsigned int*>(s_em + 15) + 1); return; }
  for (int i = threadIdx.x; i < N; i += blockDim.x) {
    const uint32_t v = hist[i];
    if (v) {
      if (p.flush_system) atomicAdd_system(&count_row[i], (unsigned long long)v);
      else atomicAdd(&count_row[i], (unsigned long long)v);
    }
  }
}

// kernel variants: hist_in_smem x fast x multi; the register bound MINB only varies for the hot FIRST_INTERACTION FAST kernel
typedef void (*TraceKernel)(const TraceParams);
static TraceKernel kernel_variant(bool hist, bool fast, int minb, bool multi, bool sq, int queue_depth = 0) {
  if (sq && hist && fast && multi) return (TraceKernel)trace_exchange_sq_kernel<4, true>;   // multi-bounce on the single-quad domain
  if (sq && hist && fast && !multi) {
    if (minb == 3) return (TraceKernel)trace_exchange_kernel<true, true, 4, false, true>;   // RTHX_MINB=3: the shared-loop form (A/B knob)
    return (TraceKernel)trace_exchange_sq_kernel<4, false>;
  }
  if (minb == 6 && hist && fast && !sq) {                                                               // per-warp ray queue (multi-face meshes; MULTI_BOUNCE on any analytic mesh)
    const bool bilin = (queue_depth & 8) != 0;                                                          // depth + 8: bilinear faces present
    const int d = queue_depth & 7;
    if (queue_depth & 16) {                                                                             // depth + 16: faces on the generic locator (FIRST_INTERACTION; compiled depths 2, 4)
      if (queue_depth & 32) return d >= 4 ? (TraceKernel)trace_exchange_queue_kernel<3, 4, true, false, true> : (TraceKernel)trace_exchange_queue_kernel<3, 2, true, false, true>;   // RTHX_GENERIC_MINB=3
      return d >= 4 ? (TraceKernel)trace_exchange_queue_kernel<4, 4, true, false, true> : (TraceKernel)trace_exchange_queue_kernel<4, 2, true, false, true>;
    }
    if (multi) {                                                                                        // compiled depths: 1, 2
      if (d >= 2) return bilin ? (TraceKernel)trace_exchange_queue_kernel<3, 2, true, true> : (TraceKernel)trace_exchange_queue_kernel<3, 2, false, true>;
      return bilin ? (TraceKernel)trace_exchange_queue_kernel<3, 1, true, true> : (TraceKernel)trace_exchange_queue_kernel<3, 1, false, true>;
    }
    if (d >= 4) return bilin ? (TraceKernel)trace_exchange_queue_kernel<4, 4, true, false> : (TraceKernel)trace_exchange_queue_kernel<4, 4, false, false>;
    if (d >= 2) return bilin ? (TraceKernel)trace_exchange_queue_kernel<4, 2, true, false> : (TraceKernel)trace_exchange_queue_kernel<4, 2, false, false>;
    return bilin ? (TraceKernel)trace_exchange_queue_kernel<4, 1, true, false> : (TraceKernel)trace_exchange_queue_kernel<4, 1, false, false>;
  }
  if (multi) {
    if (hist) return fast ? (TraceKernel)trace_exchange_kernel<true, true, 2, true, false> : (TraceKernel)trace_exchange_kernel<true, false, 2, true, false>;
    return fast ? (TraceKernel)trace_exchange_kernel<false, true, 2, true, false> : (TraceKernel)trace_exchange_kernel<false, false, 2, true, false>;
  }
  if (!hist) return fast ? (TraceKernel)trace_exchange_kernel<false, true, 2, false, false> : (TraceKernel)trace_exchange_kernel<false, false, 2, false, false>;
  if (!fast) return minb == 4 ? (TraceKernel)trace_exchange_kernel<true, false, 4, false, false>     // generic locator: 64 registers, 4 blocks per SM (default)
                              : (TraceKernel)trace_exchange_kernel<true, false, 3, false, false>;    // 80 registers, 3 blocks per SM
  switch (minb) {
    case 3: return (TraceKernel)trace_exchange_kernel<true, true, 3, false, false>;
    case 4: return (TraceKernel)trace_exchange_kernel<true, true, 4, false, false>;
    default: return (TraceKernel)trace_exchange_kernel<true, true, 2, false, false>;
  }
}

static TraceKernel hash_kernel_variant(bool fast) {
  return fast ? (TraceKernel)trace_exchange_hash_kernel<true> : (TraceKernel)trace_exchange_hash_kernel<false>;
}

cudaError_t configure_trace_kernel(size_t smem_bytes) {
  for (int sq = 0; sq < 2; ++sq)
    for (int multi = 0; multi < 2; ++multi)
      for (int hist = 0; hist < 2; ++hist)
        for (int fast = 0; fast < 2; ++fast)
          for (int minb = 2; minb <= 6; ++minb)
            for (int depth : {1, 2, 4, 9, 10, 12, 18, 20, 50, 52}) {
              cudaError_t e = cudaFuncSetAttribute((const void*)kernel_variant(hist, fast, minb, multi, sq, depth), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes);
              if (e != cudaSuccess) return e;
            }
  for (int fast = 0; fast < 2; ++fast) {
    cudaError_t e = cudaFuncSetAttribute((const void*)hash_kernel_variant(fast), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes);
    if (e != cudaSuccess) return e;
  }
  return cudaSuccess;
}

int trace_kernel_max_blocks_per_sm(int block_threads, size_t smem_bytes, bool hist, bool fast, int minb, bool multi, bool sq, int queue_depth, bool hash) {
  int n = 0;
  const void* k = hash ? (const void*)hash_kernel_variant(fast) : (const void*)kernel_variant(hist, fast, minb, multi, sq, queue_depth);
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, k, block_threads, smem_bytes) != cudaSuccess) return 0;
  return n;
}

cudaError_t launch_trace_exchange(const TraceParams& p, int n_blocks, int block_threads, size_t smem_bytes, bool fast, int minb, bool sq,
                                  cudaStream_t stream) {
  if (n_blocks <= 0) return cudaSuccess;
  TraceKernel k = p.sk_keys ? hash_kernel_variant(fast)
                            : kernel_variant(p.hist_in_smem != 0, fast, minb, p.multi_bounce != 0, sq, p.queue_depth + p.queue_bilinear);   // queue_bilinear: variant bits 8 | 16 | 32
  void* args[] = {(void*)&p};
  return cudaLaunchKernel((const void*)k, dim3(n_blocks), dim3(block_threads), args, smem_bytes, stream);
}

// ------------------------------------------------------------------------------------------------------------
// FP64 FMA-chain micro-benchmark: the measured denominator of the FP64 roofline.
// ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) fp64_peak_kernel(double* out, int iters) {
  double a0 = 1.0 + threadIdx.x * 1e-9, a1 = a0 + 1e-3, a2 = a0 + 2e-3, a3 = a0 + 3e-3;
  double a4 = a0 + 4e-3, a5 = a0 + 5e-3, a6 = a0 + 6e-3, a7 = a0 + 7e-3;
  const double m = 0.999999999, c = 1e-9;
  for (int i = 0; i < iters; ++i) {
    a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
    a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
}

cudaError_t launch_fp64_peak(double* out, int n_blocks, int block_threads, int iters, cudaStream_t stream) {
  fp64_peak_kernel<<<n_blocks, block_threads, 0, stream>>>(out, iters);
  return cudaGetLastError();
}

}  // namespace rthx
