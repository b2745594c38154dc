/* direct_fields_oracle.c — TEST INFRASTRUCTURE: method=:direct with the redirection tally (rthx_trace_direct_fields) on the CPU.
 *
 * The direct oracle (direct_oracle.c, which includes the CPU oracle whole) is included unchanged: the bundle below is traced by the
 * oracle's own emitters, traversals, event draws and MULTI_BOUNCE event rules, and re-emitted with the direct oracle's draws.  Only the
 * redirection tally and the segment count are added.  Compiled by the tests into a library of its own (tests/direct_fields_oracle.py).
 */
#include "direct_oracle.c"

/* shoot_direct of direct_oracle.c plus the redirection tally: every scattering or reflection at element k is tallied in redir[k] (no
 * draw added), and *segs grows by the traversal segments of the bundle (one per traversal, ending in an interaction or a loss).
 * Returns the element that finally absorbs the bundle (not tallied here) or -1 (lost). */
static int shoot_direct_fields(const omesh_t* o, const double* beta_all, const rthx_trace_args* a, int e, uint64_t ray_id,
                               const uint8_t* reemit, uint64_t* row, uint64_t* redir, uint64_t* segs) {
  const rthx_mesh* m = o->m;
  const int band = a->bins[0];
  const double* beta_band = beta_all + (size_t)band * m->n_cells;
  const int uniform = m->uniform_beta[band] > -0.1;
  draws_t d;
  ray_t r;
  double R_S;
  int c = o->em_coarse[e];
  {
    const poly_t* cell = &o->fine[c].faces[o->em_cell[e] - m->fine_off[c]];
    draws_init(&d, a->seed, ray_id, (uint32_t)e, (uint32_t)band, 2);
    if (e < o->ns) { r = emit_surface(cell, o->em_wall[e], a->nudge, &d); R_S = rthx_oracle_u52(d.w[4], d.w[5]); }
    else { r = emit_volume(cell, a->nudge, &d); R_S = rthx_oracle_u52(d.w[6], d.w[7]); }
  }
  hit_t h = uniform ? trace_uniform(o, r, beta_band[0], a->nudge, c, R_S) : trace_variable(o, r, beta_band, a->nudge, c, R_S);
  int n_reemit = 0;
  for (int event = 0;; ++event) {
    ++*segs;
    if (!h.ok) return -1;
    const int gh = m->fine_off[h.coarse] + h.fine;
    const int absorber = h.wall > 0 ? m->cell_surf_id[gh * 4 + (h.wall - 1)] : o->ns + gh;
    if (absorber < 0) return -1;
    if (event >= 16000) return -1;
    draws_event(&d, a->seed, ray_id, (uint32_t)e, (uint32_t)band, event);
    if (event >= 1000 && rthx_oracle_u32(d.w[3]) > 0.8) return -1;
    const double dec = rthx_oracle_u32(d.w[0]);
    ray_t r2;
    r2.px = h.px; r2.py = h.py;
    int absorbed;
    if (h.wall == 0) {
      const size_t ib = (size_t)band * m->n_cells + gh;
      const double beta = m->kappa[ib] + m->sigma_s[ib];
      const double omega = beta > 0 ? m->sigma_s[ib] / beta : 0.0;
      absorbed = !(dec < omega);
      if (!absorbed) {
        const double theta = acos(2 * rthx_oracle_u52(d.w[4], d.w[5]) - 1);
        const double phi = (2.0 * M_PI) * rthx_oracle_u32(d.w[1]);
        r2.dx = sin(theta) * cos(phi);
        r2.dy = cos(theta);
      }
    } else {
      const double eps = m->epsilon ? m->epsilon[(size_t)band * o->ns + absorber] : 1.0;
      absorbed = dec < eps;
      if (!absorbed) {
        const poly_t* cell = &o->fine[h.coarse].faces[h.fine];
        const double nx = -cell->nx[h.wall - 1], ny = -cell->ny[h.wall - 1];
        if (a->mode == RTHX_MULTI_BOUNCE_SPECULAR) {
          const double dn = r.dx * nx + r.dy * ny;
          r2.dx = r.dx - 2 * dn * nx;
          r2.dy = r.dy - 2 * dn * ny;
        } else {
          const float cosTheta = sqrtf(rthx_oracle_u23(d.w[2]));
          const float cos2 = cosTheta * cosTheta;
          const double sinTheta = sqrt(1.0 - (double)cos2);
          const double xdir = sinTheta * cos((2.0 * M_PI) * (double)rthx_oracle_u23(d.w[1]));
          const double zdir = (double)cosTheta;
          r2.dx = ny * xdir + nx * zdir;
          r2.dy = -nx * xdir + ny * zdir;
        }
      }
    }
    if (absorbed) {
      if (!reemit[absorber]) return absorber;
      row[absorber]++;                                    /* absorbed by an element of unknown temperature: emitted again from it */
      c = o->em_coarse[absorber];
      const poly_t* cell = &o->fine[c].faces[o->em_cell[absorber] - m->fine_off[c]];
      draws_reemit(&d, a->seed, ray_id, (uint32_t)e, (uint32_t)band, n_reemit++);
      if (absorber < o->ns) { r = emit_surface(cell, o->em_wall[absorber], a->nudge, &d); R_S = rthx_oracle_u52(d.w[4], d.w[5]); }
      else { r = emit_volume(cell, a->nudge, &d); R_S = rthx_oracle_u52(d.w[6], d.w[7]); }
    } else {
      redir[absorber]++;                                  /* scattered or reflected at absorber */
      r = r2;
      R_S = rthx_oracle_u52(d.w[6], d.w[7]);
      c = h.coarse;
    }
    h = uniform ? trace_uniform(o, r, beta_band[0], a->nudge, c, R_S) : trace_variable(o, r, beta_band, a->nudge, c, R_S);
  }
}

/* rthx_trace_direct_fields on the CPU, same Philox numbering: counts [n_sources][N] and lost [N] as rthx_oracle_trace_direct, plus the
 * redirection counts redirected [n_sources][N] (row y = source sources[y], every scattering or reflection of its bundles at element k
 * in column k) and *segments_out, the traversal segments of all bundles (the device's events_out). */
int rthx_oracle_trace_direct_fields(const rthx_mesh* m, const rthx_trace_args* a, const int32_t* sources, const int64_t* rays, int32_t n_sources,
                                    const uint8_t* reemit, uint64_t* counts, uint64_t* redirected, uint64_t* lost, uint64_t* segments_out,
                                    int n_threads) {
  if (check_args(m, a) || a->n_bins != 1 || !counts || !redirected || !sources || !rays || !reemit || n_sources < 1) return RTHX_ERR_ARG;
  if (a->mode != RTHX_MULTI_BOUNCE && a->mode != RTHX_MULTI_BOUNCE_SPECULAR) return RTHX_ERR_ARG;
  if (g_faithful) return RTHX_ERR_ARG;
  omesh_t o;
  const int rc = omesh_build(&o, m);
  if (rc) { omesh_free(&o); return rc == 1 ? RTHX_ERR_NOMEM : RTHX_ERR_ARG; }
  const int N = o.N;
  for (int32_t y = 0; y < n_sources; ++y)
    if (sources[y] < 0 || sources[y] >= N) { omesh_free(&o); return RTHX_ERR_ARG; }
  double* beta_all = (double*)malloc(sizeof(double) * (size_t)m->n_bands * m->n_cells);
  for (size_t i = 0; i < (size_t)m->n_bands * m->n_cells; ++i) beta_all[i] = m->kappa[i] + m->sigma_s[i];
  memset(counts, 0, sizeof(uint64_t) * (size_t)n_sources * N);
  memset(redirected, 0, sizeof(uint64_t) * (size_t)n_sources * N);
  if (lost) memset(lost, 0, sizeof(uint64_t) * (size_t)N);
  uint64_t segments = 0;
#ifdef _OPENMP
  if (n_threads > 0) omp_set_num_threads(n_threads);
#else
  (void)n_threads;
#endif
#pragma omp parallel for schedule(dynamic, 1) reduction(+ : segments)
  for (int32_t y = 0; y < n_sources; ++y) {
    const int e = sources[y];
    uint64_t* row = counts + (size_t)y * N;
    uint64_t* red = redirected + (size_t)y * N;
    uint64_t nlost = 0;
    for (int64_t i = 0; i < rays[y]; ++i) {
      const int ab = shoot_direct_fields(&o, beta_all, a, e, (uint64_t)(a->ray_id_offset + i), reemit, row, red, &segments);
      if (ab < 0) nlost++; else row[ab]++;
    }
    if (lost) lost[e] = nlost;
  }
  if (segments_out) *segments_out = segments;
  free(beta_all);
  omesh_free(&o);
  return RTHX_OK;
}
