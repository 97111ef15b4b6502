/*
 * repair_oracle.c -- CPU restatement of the checked solve's pieces (cfs_solve_batch_margins, the repair increments of
 * cfs_solve_checked; include/cfs_b200.h).  TEST INFRASTRUCTURE, never linked into libcfs_b200.so.
 *
 * Compiled as the tail of a copy of oracle/cfs_oracle.c in which the obstacle row's "I = distance - c->margin[j]" reads
 * "distance - (c->margin[j] + off)" when the thread's offset pointer orc_moff is set (tests/repair_oracle.py makes that copy
 * and refuses to build when the line is not found exactly once).  With orc_moff == NULL the copy evaluates exactly the
 * oracle's expression, so it reproduces every golden bit for bit.  Same flags as the oracle (-O2 -ffp-contract=off).
 */

#define REPAIR_MAXOBS 32

/* orc_cfs_solve_batch2 with per-waypoint offsets moff (nobs x H per problem, [prob][obs][i]; NULL = none) */
void orc_cfs_solve_batch_off(const orc_robot *r, const orc_cfg *c, int B, int nthreads, const double *x0, const double *ff,
                             const double *caug, const double *xref, const double *noise, const double *moff, double *u,
                             double *x, double *cost_hist, double *e_u_hist, int *iters, int *status) {
  const int nj = r->nj, ns = 2 * nj, H = c->H, n = nj * H, N = ns * H;
  double *J0 = NULL;
  if (c->solver == 0) {
    J0 = (double *)malloc(sizeof(double) * n * n);
    if (orc_chol_J0(n, c->QQ, J0)) {
      for (int b = 0; b < B; ++b) {
        status[b] = ORC_NUMERICAL;
        iters[b] = 0;
      }
      free(J0);
      return;
    }
  }
#ifdef _OPENMP
  if (nthreads > 0) omp_set_num_threads(nthreads);
#endif
  (void)nthreads;
#pragma omp parallel for schedule(dynamic, 1)
  for (int b = 0; b < B; ++b) {
    for (int k = 0; k < c->max_outer; ++k) cost_hist[(size_t)b * c->max_outer + k] = NAN;
    if (e_u_hist)
      for (int k = 0; k < c->max_outer; ++k) e_u_hist[(size_t)b * c->max_outer + k] = NAN;
    orc_moff = moff ? moff + (size_t)b * c->nobs * H : NULL;
    status[b] = orc_cfs_solve(r, c, J0, x0 + (size_t)b * ns, ff + (size_t)b * n, caug[b], xref + (size_t)b * N,
                              noise ? noise + (size_t)b * n * c->max_outer : NULL, u + (size_t)b * n, x + (size_t)b * N,
                              cost_hist + (size_t)b * c->max_outer, e_u_hist ? e_u_hist + (size_t)b * c->max_outer : NULL,
                              &iters[b], NULL);
    orc_moff = NULL;
  }
  if (J0) free(J0);
}

/* The repair increments of k_repair_margins (csrc/k_repair.cu) for B trajectories: segments in order; HIT segment k
 * (seg_verdict[b H + k] == 1): witness theta* = (theta_k + omega_k s) + ((0.5 s) s) u_k at s = seg_s_hit[b H + k], per obstacle
 * c_j = dist_arm(theta*, obs_j) - m_j, inc_j = gain (eta - c_j) where c_j < -eta/2; waypoint i in 1..H gets
 * max(inc of segment i-1, inc of segment i), added to off[(b nobs + j) H + i - 1]. */
void orc_repair_increments(const orc_robot *r, int nobs, const double *obs, const double *margin, int B, int H, const double *x0,
                           const double *x, const double *u, const int *seg_verdict, const double *seg_s_hit, double eta,
                           double gain, double *off) {
  const int nj = r->nj;
  const double half_eta = 0.5 * eta;
  for (int b = 0; b < B; ++b) {
    double prev[REPAIR_MAXOBS], cur[REPAIR_MAXOBS];
    for (int j = 0; j < nobs; ++j) prev[j] = 0.0;
    double *ob = off + (size_t)b * nobs * H;
    for (int k = 0; k < H; ++k) {
      const size_t it = (size_t)b * H + k;
      for (int j = 0; j < nobs; ++j) cur[j] = 0.0;
      if (seg_verdict[it] == 1) {
        const double *p0 = k == 0 ? x0 + (size_t)b * 2 * nj : x + ((size_t)b * H + (k - 1)) * 2 * nj;
        const double *p1 = p0 + nj, *pu = u + it * nj;
        const double s = seg_s_hit[it];
        double th[ORC_MAXL];
        for (int q = 0; q < nj; ++q) th[q] = (p0[q] + p1[q] * s) + ((0.5 * s) * s) * pu[q];
        for (int j = 0; j < nobs; ++j) {
          const double c = orc_dist_arm(r, th, obs + ORC_OBS_STRIDE * j, NULL, NULL) - margin[j];
          if (c < -half_eta) cur[j] = gain * (eta - c);
        }
      }
      if (k > 0)
        for (int j = 0; j < nobs; ++j) ob[(size_t)j * H + (k - 1)] += prev[j] > cur[j] ? prev[j] : cur[j];
      for (int j = 0; j < nobs; ++j) prev[j] = cur[j];
    }
    for (int j = 0; j < nobs; ++j) ob[(size_t)j * H + (H - 1)] += prev[j];
  }
}
