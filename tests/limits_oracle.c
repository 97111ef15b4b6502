/* Joint position limits on the CPU restatement (cfs_set_joint_limits, include/cfs_b200.h).  TEST INFRASTRUCTURE.
 *
 * Compiled as the tail of a copy of oracle/cfs_oracle.c (tests/limits_oracle.py) whose orc_cfs_solve appends, when orc_qlim is
 * set, the 2n constant rows after the bound rows: for waypoint i = 1..H and joint k (e = (i-1) nj + k)
 *   row m0 + e:      B_theta(e, :) u <= qmax_k - fm,     row m0 + n + e:  -B_theta(e, :) u <= fm - qmin_k,
 * with the free motion fm = theta0_k + (i dt) omega0_k and B_theta(e, (jj-1) nj + k) = (0.5 + (i - jj)) dt^2 for jj <= i. */

static void orc_limit_rows(int nj, int H, double dt, const double *x0, const double *qlim /* qmin (nj) | qmax (nj) */,
                           double *A /* 2n x n row-major */, double *b) {
  const int n = nj * H;
  for (int e = 0; e < n; ++e) {
    const int i = e / nj, k = e - i * nj; /* waypoint i + 1 */
    double *up = A + (size_t)e * n, *dn = A + (size_t)(n + e) * n;
    for (int c = 0; c < n; ++c) up[c] = dn[c] = 0.0;
    for (int jj = 0; jj <= i; ++jj) {
      const double v = 0.5 * dt * dt + ((i - jj) * dt) * dt;
      up[jj * nj + k] = v;
      dn[jj * nj + k] = -v;
    }
    const double fm = x0[k] + ((i + 1) * dt) * x0[nj + k];
    b[e] = qlim[nj + k] - fm;
    b[n + e] = fm - qlim[k];
  }
}

/* orc_cfs_solve_batch2 with joint limits qlim (NULL = none) */
void orc_cfs_solve_batch_lim(const orc_robot *r, const orc_cfg *c, int B, int nthreads, const double *x0, const double *ff,
                             const double *caug, const double *xref, const double *noise, const double *qlim, double *u,
                             double *x, double *cost_hist, double *e_u_hist, int *iters, int *status, int *qp_stats) {
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
    orc_qlim = qlim;
    status[b] = orc_cfs_solve(r, c, J0, x0 + (size_t)b * ns, ff + (size_t)b * n, caug[b], xref + (size_t)b * N,
                              noise ? noise + (size_t)b * n * c->max_outer : NULL, u + (size_t)b * n, x + (size_t)b * N,
                              cost_hist + (size_t)b * c->max_outer, e_u_hist ? e_u_hist + (size_t)b * c->max_outer : NULL,
                              &iters[b], qp_stats ? qp_stats + 2 * b : NULL);
    orc_qlim = NULL;
  }
  if (J0) free(J0);
}

/* orc_get_con followed by the 2n limit rows (Ainq row-major, m + 2n rows); returns the row count */
int orc_get_con_lim(const orc_robot *r, const orc_cfg *c, const double *x0, const double *xcur, const double *u,
                    const double *qlim, double *Ainq, double *binq) {
  const int n = r->nj * c->H;
  int touched = 0;
  const int m = orc_get_con(r, c, x0, xcur, u, Ainq, binq, NULL, NULL, NULL, &touched);
  if (!qlim) return m;
  orc_limit_rows(r->nj, c->H, r->dt, x0, qlim, Ainq + (size_t)m * n, binq + m);
  return m + 2 * n;
}
