// rthx_trace_body.cuh — body of K1 (rthx_kernels.cu), shared by trace_exchange_kernel<HIST_SMEM, FAST, MINB, MULTI, SQ> and
// trace_exchange_hash_kernel<FAST>.  It is included INSIDE their function bodies, where HIST_SMEM, FAST, MULTI, SQ and HASH
// are compile-time constants and `p` is the __grid_constant__ parameter: inlining it through a device function taking the
// parameter by reference changed the code ptxas generates for the existing instances, textual inclusion does not.
  extern __shared__ __align__(16) unsigned char smem_raw[];
  CoarseDev* s_coarse = reinterpret_cast<CoarseDev*>(smem_raw);
  const bool coarse_smem = !SQ && (FAST || p.coarse_in_smem);
  const size_t coarse_bytes = coarse_smem ? sizeof(CoarseDev) * (size_t)p.n_coarse : 0;
  double* s_em = reinterpret_cast<double*>(smem_raw + coarse_bytes);
  double2* s_log = reinterpret_cast<double2*>(smem_raw + coarse_bytes + sizeof(double) * EM_DOUBLES);
  uint32_t* hist = reinterpret_cast<uint32_t*>(smem_raw + coarse_bytes + sizeof(double) * EM_DOUBLES + sizeof(double2) * LOGTAB_N);

  // block -> (owned emitter ordinal y, traced bin bi, ray chunk)
  const unsigned bid = blockIdx.x;
  const int chunk = (int)(bid % (unsigned)p.row_chunks);
  const unsigned t1 = bid / (unsigned)p.row_chunks;
  const int bi = (int)(t1 % (unsigned)p.n_bins);
  const int y = p.y_offset + (int)(t1 / (unsigned)p.n_bins);
  const int e = p.emitter_rank + y * p.emitter_world;
  const int band = p.bins[bi];
  const int N = p.N;

  // stage coarse faces and the emitter description, clear the row histogram
  if (coarse_smem) {
    const int nw = (int)(coarse_bytes / 8);
    const double* src = reinterpret_cast<const double*>(p.coarse);
    double* dst = reinterpret_cast<double*>(s_coarse);
    for (int i = threadIdx.x; i < nw; i += blockDim.x) dst[i] = src[i];
  }
  if (HIST_SMEM)
    for (int i = threadIdx.x; i < N; i += blockDim.x) hist[i] = 0u;
  if (HASH)
    for (int i = threadIdx.x; i < (2 << p.sk_slots_log2) + 2; i += blockDim.x) hist[i] = 0u;
  for (int i = threadIdx.x; i < LOGTAB_N; i += blockDim.x) s_log[i] = c_logtab[i];
  // FAST: a plain shared-memory pointer (LDS); otherwise a generic pointer that may be shared or global
  const CoarseDev* coarse = FAST ? s_coarse : (p.coarse_in_smem ? s_coarse : p.coarse);

  const int g = p.em_cell[e];
  const int wall = p.em_wall[e];
  const int c0 = p.em_coarse[e];
  const bool is_surface = wall >= 0;
  const int em_nv = p.poly_nv[g];
  if (threadIdx.x == 0) {
    const double* vx = p.poly_vx + 4 * g;
    const double* vy = p.poly_vy + 4 * g;
    if (is_surface) {
      const int j = (wall + 1 == em_nv) ? 0 : wall + 1;
      const double ex = vx[j] - vx[wall], ey = vy[j] - vy[wall];
      const double len = sqrt(ex * ex + ey * ey);
      s_em[0] = vx[wall]; s_em[1] = vy[wall]; s_em[2] = ex; s_em[3] = ey;
      s_em[4] = ex / len; s_em[5] = ey / len;       // xVecLocal
      s_em[6] = -(ey / len); s_em[7] = ex / len;    // yVecLocal
    } else {
      s_em[0] = vx[0]; s_em[1] = vy[0]; s_em[2] = vx[1] - vx[0]; s_em[3] = vy[1] - vy[0]; s_em[4] = vx[2] - vx[0]; s_em[5] = vy[2] - vy[0];
      s_em[6] = vx[2]; s_em[7] = vy[2]; s_em[8] = vx[3] - vx[2]; s_em[9] = vy[3] - vy[2]; s_em[10] = vx[0] - vx[2]; s_em[11] = vy[0] - vy[2];
      // emitVolumeRay2D.jl:7 — area(ABC)/volume; triangles always take the first (only) triangle
      s_em[14] = em_nv == 3 ? 2.0 : 0.5 * (vx[0] * (vy[1] - vy[2]) + vx[1] * (vy[2] - vy[0]) + vx[2] * (vy[0] - vy[1])) / p.cell_volume[g];
    }
    s_em[12] = p.cell_mid[2 * g]; s_em[13] = p.cell_mid[2 * g + 1];
  }

  // ray range of this chunk
  const int64_t per = (p.rays_per_emitter + p.row_chunks - 1) / p.row_chunks;
  const int64_t r_begin = (int64_t)chunk * per;
  int64_t r_end = r_begin + per;
  if (r_end > p.rays_per_emitter) r_end = p.rays_per_emitter;

  const double ub = p.uniform_beta[band];
  const bool uniform = ub > -0.1;                      // traceRay.jl:4
  const double* beta_band = p.beta + (size_t)band * p.n_cells;
  const double beta_u = beta_band[0];                  // traceRay.jl:6-11: beta of fine_mesh[1][1]
  const double inv_beta_u = beta_u > 0.0 ? 1.0 / beta_u : CUDART_INF;
  const int rec_slot = (p.rec_slot != nullptr && band == p.rec_bin) ? p.rec_slot[e] : -1;
  const size_t row = p.compact_rows ? ((size_t)bi * p.n_owned + y) : ((size_t)bi * N + e);
  unsigned long long* count_row = p.counts + row * (size_t)N;

  __syncthreads();

  const uint32_t cw = ((uint32_t)band << 16);
  unsigned int n_lost = 0;
  const unsigned long long row_key = HASH ? (unsigned long long)y * (unsigned long long)p.n_bins + (unsigned long long)bi : 0ull;

  // HASH: block-synchronous rounds (every thread runs every round; lanes past r_end only take part in the flush)
  for (int64_t r = r_begin + threadIdx.x; HASH ? r - (int64_t)threadIdx.x < r_end : r < r_end; r += blockDim.x) {
    if constexpr (HASH) {
      const uint32_t S = 1u << p.sk_slots_log2;
      __syncthreads();
      const bool flush = hist[2 * S] + blockDim.x > S / 2;   // the coming round could pass half full
      __syncthreads();
      if (flush && !hash_flush(p, hist, row_key)) return;
      if (r >= r_end) continue;
    }
    const uint64_t ray_id = (uint64_t)(p.ray_id_offset + r);
    const uint32_t c_lo = (uint32_t)ray_id, c_hi = (uint32_t)(ray_id >> 32);
    // two Philox calls per ray: w0 (call 0) feeds the emission point/azimuth, w1 (call 1) the 52-bit draws
    const uint4 w0 = philox4x32_10_rk(make_uint4(c_lo, c_hi, (uint32_t)e, cw | 0u), p.rk);
    const uint4 w1 = philox4x32_10_rk(make_uint4(c_lo, c_hi, (uint32_t)e, cw | 1u), p.rk);
    double px, py, dx, dy, R_S;
    // ---- stage 1: emission --------------------------------------------------------------------------------
    if (is_surface) {
      const double R = u32d(w0.x, p.k_u32);
      px = fma(s_em[2], R, s_em[0]);
      py = fma(s_em[3], R, s_em[1]);
      // lambertSample2D: Float32 variates / sqrt / square, the rest in Float64
      const float cosT = __fsqrt_rn(u23(w0.y));
      const float cos2 = __fmul_rn(cosT, cosT);
      const double sinT = sqrt_pos(1.0 - (double)cos2);
      const double xdir = sinT * cos2pi_unit((double)u23(w0.z));
      const double zdir = (double)cosT;
      dx = s_em[4] * xdir + s_em[6] * zdir;
      dy = s_em[5] * xdir + s_em[7] * zdir;
      R_S = u52(w1.x, w1.y, p.k_u52);
    } else {
      const double R1 = u32d(w0.x, p.k_u32), R2 = u32d(w0.y, p.k_u32);
      const double sq = sqrt_pos(R1);
      // uniform point of triangle (V0,V1,V2): V0 + sqrt(R1)(1-R2)(V1-V0) + sqrt(R1) R2 (V2-V0), emitVolumeRay2D.jl:9,12
      const double* tri = s_em + ((u32d(w0.z, p.k_u32) < s_em[14]) ? 0 : 6);
      const double a2 = sq * R2, a1 = sq - a2;
      px = fma(a2, tri[4], fma(a1, tri[2], tri[0]));
      py = fma(a2, tri[5], fma(a1, tri[3], tri[1]));
      // theta = acos(1-2R): cos(theta) = 1-2R, sin(theta) = 2 sqrt(R(1-R)) (algebraically identical)
      const double Rt = u52(w1.x, w1.y, p.k_u52);
      const double sinT = 2.0 * sqrt_pos(Rt * (1.0 - Rt));
      const double phiR = u32d(w0.w, p.k_u32);
      dx = sinT * cos2pi_unit(phiR);
      dy = fma(Rt, -2.0, 1.0);
      R_S = u52(w1.z, w1.w, p.k_u52);
    }
    px = fma(s_em[12] - px, p.nudge, px);   // nudge towards the cell midpoint (emitSurfaceRay2D.jl:10, emitVolumeRay2D.jl:22)
    py = fma(s_em[13] - py, p.nudge, py);
    if (rec_slot >= 0) {                    // RayRecorder origin (kept only if the ray is tallied: rec_valid below)
      double* o = p.rec_pts + 4 * ((size_t)rec_slot * (size_t)p.rays_per_emitter + (size_t)r);
      o[0] = px; o[1] = py;
    }

    // ---- stage 2: first-interaction traversal (traceRayUniform / traceRayVariable) --------------------------
    // MULTI (RTHX_MULTI_BOUNCE): the traversal is repeated from every scattering / reflection event until the ray is
    // absorbed (traceSingleRay.jl:7-81 without the re-emission branches); otherwise the body runs exactly once.
    double neg_log = neg_log_table(R_S, s_log);
    int c = c0;
    int absorber = -1;
    if constexpr (SQ) {
      // single parallelogram face: one distToSurface2D, one decision, one fine-cell location (traceRay.jl:27-52)
      const CoarseDev& cf = p.face0;
      int k;
      const double u = dist_quad(cf, px, py, dx, dy, p.k_eps, k);
      double S = neg_log * inv_beta_u;
      bool gas = S < u, ok = true;
      if (!uniform) {
        const int f0 = locate_quad(cf, px, py);              // traceRay.jl:87-100
        ok = f0 >= 0;
        const double local_beta = ok ? beta_band[f0] : 0.0;
        gas = local_beta * u >= neg_log;
        S = neg_log / local_beta;
      }
      // Gas and wall endings share one advance + one fine-cell location (same arithmetic as the two branches of
      // traceRay.jl:31-52, selected per lane): a warp with both kinds of ray no longer issues the tail twice.
      const bool hit = !gas & (u < CUDART_INF) & (cf.solid[k] != 0);   // an open edge has no neighbour face: the ray is lost
      if (ok & (gas | hit)) {
        const double adv = (gas ? S : u) - p.nudge;
        px = fma(adv, dx, px);
        py = fma(adv, dy, py);
        const int f = locate_quad(cf, px, py);
        if (f >= 0) absorber = gas ? p.n_surfaces + f : __ldg(p.cell_surf_id + 4 * f + k);
      }
    } else {
    double hit_nx = 0.0, hit_ny = 0.0;   // MULTI: outward unit normal of the wall that was hit
#pragma unroll 1
    for (int event = 0;; ++event) {
    double S = uniform ? neg_log * inv_beta_u : 0.0;   // remaining free path (uniform); beta = 0 -> Inf
    double acc = 0.0;                                  // accumulated tau (variable)
    absorber = -1;
    for (int it = 0; it < 10000; ++it) {
      const CoarseDev& cf = coarse[c];
      const int kind = FAST ? cf.kind : ((p.force_generic || cf.kind == KIND_BILINEAR_QUAD) ? KIND_GENERIC : cf.kind);   // the bilinear inverse lives in the queue kernel only
      int k;
      const double u = FAST ? dist_fast(cf, px, py, dx, dy, p.k_eps, k) : dist_to_coarse(cf, px, py, dx, dy, p.k_eps, k);
      bool gas;
      double tau_b = 0.0;
      if (uniform) {
        gas = S < u;
      } else {
        const int f0 = locate_fine<FAST>(p, cf, c, kind, px, py);   // traceRay.jl:87-100
        if (f0 < 0) break;
        const double local_beta = beta_band[cf.fine_off + f0];
        tau_b = local_beta * u;
        gas = acc + tau_b >= neg_log;
        if (gas) S = (neg_log - acc) / local_beta;
      }
      // Gas events and solid-wall hits share ONE advance and ONE fine-cell location (the same arithmetic as the two branches of
      // traceRay.jl:31-52, selected per lane): with separate call sites a warp holding both kinds of ray ran the point location —
      // the expensive part of the generic locator — twice at half occupancy (ncu: 2.0 calls per warp and ray at 16 lanes).
      const bool noedge = !(u < CUDART_INF);
      if (!gas & noedge) break;                                   // no edge ahead: the reference ends in NaN -> lost
      const bool solid = !gas && cf.solid[k];
      const double adv = gas ? S - p.nudge : (solid ? u - p.nudge : u + p.nudge);   // traceRay.jl:33,44,56
      px = fma(adv, dx, px);
      py = fma(adv, dy, py);
      if (gas | solid) {
        const int f = locate_fine<FAST>(p, cf, c, kind, px, py);
        if (f < 0) break;
        const int gc = cf.fine_off + f;
        if (gas) { absorber = p.n_surfaces + gc; break; }
        int w;
        if (!FAST && kind == KIND_GENERIC) {
          w = wall_of_rec(p.face_rec + 12 * (size_t)gc, px, py, dx, dy, absorber);   // traceRay.jl:51; absorber -1: fine wall not solid -> lost
          if (MULTI) { hit_nx = p.poly_nx[4 * gc + w]; hit_ny = p.poly_ny[4 * gc + w]; }
          break;
        } else {
          if (MULTI) { hit_nx = cf.nx[k]; hit_ny = cf.ny[k]; }  // fine walls on a coarse edge share its normal
          if (kind == KIND_AFFINE_QUAD) {
            w = k;                                              // fine wall lying on coarse edge k
          } else if (__ldg(p.poly_nv + gc) == 3) {
            w = k;                                              // diagonal triangle cell: walls follow the coarse edges
          } else {
            if (k == cf.diag) break;
            w = (k < cf.diag) ? k : k + 1;                      // quad cell of a mirrored-triangle lattice
          }
        }
        absorber = __ldg(p.cell_surf_id + 4 * gc + w);          // -1: fine wall not solid -> lost
        break;
      } else {
        if (uniform) S -= u; else acc += tau_b;
        int nc;
        if (FAST) {
          nc = cf.nbr[k];
        } else {
          nc = (kind == KIND_GENERIC) ? -1 : cf.nbr[k];
          if (nc < 0) nc = find_face_generic(p, 0, px, py);     // traceRay.jl:59-65
        }
        if (nc < 0) break;
        c = nc;
      }
    }
    if (!MULTI || absorber < 0) break;
    // ---- MULTI_BOUNCE: absorb, scatter or reflect (traceSingleRay.jl:24-79) ---------------------------------------
    // two more Philox calls per event: call# 2+2*event (+1).  v0.x decision, v0.y azimuth / psi, v0.z cos-theta (walls),
    // v0.w roulette, (v1.x,v1.y) polar angle (gas), (v1.z,v1.w) next free path
    if (event >= 16000) { absorber = -1; break; }                // call# is a 16-bit field
    const uint4 v0 = philox4x32_10_rk(make_uint4(c_lo, c_hi, (uint32_t)e, cw | (uint32_t)(2 + 2 * event)), p.rk);
    const uint4 v1 = philox4x32_10_rk(make_uint4(c_lo, c_hi, (uint32_t)e, cw | (uint32_t)(3 + 2 * event)), p.rk);
    if (event >= 1000 && u32d(v0.w, p.k_u32) > 0.8) { absorber = -1; break; }   // Russian roulette, traceSingleRay.jl:11
    const double dec = u32d(v0.x, p.k_u32);
    if (absorber >= p.n_surfaces) {
      if (!(dec < p.omega[(size_t)band * p.n_cells + (absorber - p.n_surfaces)])) break;   // absorbed in the gas
      // isotropicScatter2D.jl:1-4: theta = acos(2R-1), phi = 2 pi R
      const double Rt = u52(v1.x, v1.y, p.k_u52);
      const double sinT = 2.0 * sqrt(Rt * (1.0 - Rt));
      dx = sinT * cospi(2.0 * u32d(v0.y, p.k_u32));
      dy = fma(Rt, 2.0, -1.0);
    } else {
      if (dec < p.eps[(size_t)band * p.n_surfaces + absorber]) break;                       // absorbed by the wall
      if (p.specular) {
        const double dn = dx * hit_nx + dy * hit_ny;            // mirror the in-plane components; the axial one is unchanged
        dx = fma(-2.0 * dn, hit_nx, dx);
        dy = fma(-2.0 * dn, hit_ny, dy);
      } else {
        // diffuse: Lambert about the inward normal n = -hit_n with x-axis (n.y, -n.x) (sampleReflectionDirection2D.jl:5-16)
        const float cosT = __fsqrt_rn(u23(v0.z));
        const float cos2 = __fmul_rn(cosT, cosT);
        const double xdir = sqrt(1.0 - (double)cos2) * cospi(2.0 * (double)u23(v0.y));
        const double zdir = (double)cosT;
        const double nxi = -hit_nx, nyi = -hit_ny;
        dx = nyi * xdir + nxi * zdir;
        dy = -nxi * xdir + nyi * zdir;
      }
    }
    neg_log = -log(u52(v1.z, v1.w, p.k_u52));
    }
    }

    // ---- stage 3/4: tally (+ record) -------------------------------------------------------------------------
    if (absorber >= 0) {
      if (HIST_SMEM) atomicAdd(&hist[absorber], 1u);
      else if (HASH) hash_insert(hist, p.sk_slots_log2, absorber);
      else if (p.flush_system) atomicAdd_system(&count_row[absorber], 1ULL);
      else atomicAdd(&count_row[absorber], 1ULL);
      if (rec_slot >= 0) {
        const size_t s = (size_t)rec_slot * (size_t)p.rays_per_emitter + (size_t)r;
        double* o = p.rec_pts + 4 * s;
        o[2] = px; o[3] = py;
        p.rec_valid[s] = 1;
      }
    } else {
      ++n_lost;
    }
  }

  // ---- flush --------------------------------------------------------------------------------------------------
  if (HASH && !hash_flush(p, hist, row_key)) return;
  for (int off = 16; off > 0; off >>= 1) n_lost += __shfl_down_sync(0xffffffffu, n_lost, off);
  if ((threadIdx.x & 31) == 0 && n_lost) {
    if (p.flush_system) atomicAdd_system(&p.lost[(size_t)bi * N + e], (unsigned long long)n_lost);
    else atomicAdd(&p.lost[(size_t)bi * N + e], (unsigned long long)n_lost);
  }
  if (HIST_SMEM) {
    __syncthreads();
    if (p.peer_counts != nullptr) { handover_row_hist(p, hist, reinterpret_cast<unsigned int*>(s_em + 15) + 1); return; }
    for (int i = threadIdx.x; i < N; i += blockDim.x) {
      const uint32_t v = hist[i];
      if (v) {
        if (p.flush_system) atomicAdd_system(&count_row[i], (unsigned long long)v);   // red.sys: matrix lives on a peer GPU
        else atomicAdd(&count_row[i], (unsigned long long)v);                          // red.gpu.global.add.u64, result unused
      }
    }
  }
