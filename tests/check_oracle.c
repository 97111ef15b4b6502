/*
 * check_oracle.c -- CPU restatement of the continuous collision checks (cfs_check_edges / cfs_check_trajectories,
 * include/cfs_b200.h).  TEST INFRASTRUCTURE, never linked into libcfs_b200.so.
 *
 * Built together with oracle/cfs_oracle.c into one shared library (tests/check_oracle.py), with the oracle's flags
 * (-O2 -ffp-contract=off): the clearance is the oracle's dist_arm per obstacle, and the motion bound, the paths, vmax and the
 * step rule are the same operations in the same order as motion_bound (csrc/cfs_api.cu) and k_check (csrc/k_check.cu).
 */
#include <math.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#include "cfs_oracle.h"

enum { CHK_CLEAR = 0, CHK_HIT = 1, CHK_UNDECIDED = 2 };

/* the per-link translations of the DH / 2L chains as the library's LinkTab holds them (cfs_set_robot) */
static void link_trans(const orc_robot *r, int i, double *a, double *fix) {
  if (r->kind == ORC_2L) {
    const int c = i + 1 < 3 ? i + 1 : 2; /* robot.T(:, i+1) */
    const double tx = r->T2L[c][0], ty = r->T2L[c][1], dz = r->T2L[c][2];
    *a = 0.0;
    *fix = sqrt((tx * tx + ty * ty) + dz * dz);
  } else {
    const double dz = r->DH[i][1];
    *a = r->DH[i][2];
    *fix = sqrt((0.0 * 0.0 + 0.0 * 0.0) + dz * dz);
  }
}

/* R[j] >= ||dp/dtheta_j|| for every link-axis endpoint p of the links l >= j (include/cfs_b200.h, "Motion bound") */
void orc_motion_bound(const orc_robot *r, double *R) {
  for (int j = 0; j < ORC_MAXL; ++j) R[j] = 0.0;
  for (int j = 0; j < r->nj; ++j) {
    double aj, fj;
    link_trans(r, j, &aj, &fj);
    double reach = fabs(aj);
    for (int l = j; l < r->nj; ++l) {
      double al, fl;
      link_trans(r, l, &al, &fl);
      if (l > j) reach = reach + (fabs(al) + fl);
      for (int k = 0; k < 2; ++k) {
        const double *cp = r->cap[l][k];
        const double c = sqrt((cp[0] * cp[0] + cp[1] * cp[1]) + cp[2] * cp[2]);
        if (reach + c > R[j]) R[j] = reach + c;
      }
    }
  }
}

/* c(theta) = min_j (dist_arm(theta, obs_j) - m_j) */
double orc_clearance(const orc_robot *r, int nobs, const double *obs, const double *margin, const double *theta) {
  double c = INFINITY;
  for (int j = 0; j < nobs; ++j) {
    const double v = orc_dist_arm(r, theta, obs + ORC_OBS_STRIDE * j, NULL, NULL) - margin[j];
    if (v < c) c = v;
  }
  return c;
}

void orc_clearance_batch(const orc_robot *r, int nobs, const double *obs, const double *margin, int N, const double *theta,
                         double *c) {
#pragma omp parallel for schedule(static)
  for (int i = 0; i < N; ++i) c[i] = orc_clearance(r, nobs, obs, margin, theta + (long)i * r->nj);
}

/* one item: mode 0 edge (p0 = theta_a, p1 = theta_b, send = 1), mode 1 segment (p0 = theta_k, p1 = omega_k, pu = u_k, send = dt) */
static int check_item(const orc_robot *r, int nobs, const double *obs, const double *margin, const double *R, int mode,
                      const double *p0, const double *p1, const double *pu, double eta, int max_evals, double *s_hit,
                      double *cmin, int *evals) {
  const int nj = r->nj;
  const double dt = r->dt, half_eta = 0.5 * eta, send = mode == 0 ? 1.0 : dt;
  double vmax = 0.0;
  for (int k = 0; k < nj; ++k) {
    double w;
    if (mode == 0) {
      w = fabs(p1[k] - p0[k]);
    } else {
      const double w0 = fabs(p1[k]), w1 = fabs(p1[k] + pu[k] * dt);
      w = w0 > w1 ? w0 : w1;
    }
    vmax = vmax + R[k] * w;
  }
  double s = 0.0, cm = INFINITY, th[ORC_MAXL];
  int ev = 0, verdict = CHK_UNDECIDED;
  *s_hit = -1.0;
  while (ev < max_evals) {
    for (int k = 0; k < nj; ++k)
      th[k] = mode == 0 ? p0[k] + s * (p1[k] - p0[k]) : (p0[k] + p1[k] * s) + ((0.5 * s) * s) * pu[k];
    const double c = orc_clearance(r, nobs, obs, margin, th);
    ++ev;
    if (c < cm) cm = c;
    if (c < -half_eta) {
      verdict = CHK_HIT;
      *s_hit = s;
      break;
    }
    if (s == send || vmax == 0.0) {
      verdict = CHK_CLEAR;
      break;
    }
    s = s + (c + eta) / vmax;
    if (!(s < send)) s = send;
  }
  *cmin = cm;
  if (evals) *evals = ev;
  return verdict;
}

int orc_check_edge(const orc_robot *r, int nobs, const double *obs, const double *margin, const double *R, const double *ta,
                   const double *tb, double eta, int max_evals, double *s_hit, double *cmin, int *evals) {
  return check_item(r, nobs, obs, margin, R, 0, ta, tb, NULL, eta, max_evals, s_hit, cmin, evals);
}

/* segment from state xk (theta_k; omega_k) with control uk over tau in [0, r->dt] */
int orc_check_segment(const orc_robot *r, int nobs, const double *obs, const double *margin, const double *R, const double *xk,
                      const double *uk, double eta, int max_evals, double *tau_hit, double *cmin, int *evals) {
  return check_item(r, nobs, obs, margin, R, 1, xk, xk + r->nj, uk, eta, max_evals, tau_hit, cmin, evals);
}

void orc_check_edges_batch(const orc_robot *r, int nobs, const double *obs, const double *margin, int N, const double *ta,
                           const double *tb, double eta, int max_evals, int *verdict, double *s_hit, double *cmin, int *evals) {
  double R[ORC_MAXL];
  orc_motion_bound(r, R);
#pragma omp parallel for schedule(dynamic, 16)
  for (int i = 0; i < N; ++i)
    verdict[i] = orc_check_edge(r, nobs, obs, margin, R, ta + (long)i * r->nj, tb + (long)i * r->nj, eta, max_evals, &s_hit[i],
                                &cmin[i], &evals[i]);
}

/* x0 (2nj x B), x (2njH x B), u (njH x B): per trajectory the reduction of include/cfs_b200.h */
void orc_check_trajectories_batch(const orc_robot *r, int nobs, const double *obs, const double *margin, int B, int H,
                                  const double *x0, const double *x, const double *u, double eta, int max_evals, int *verdict,
                                  double *t_hit, double *cmin, int *evals) {
  const int nj = r->nj;
  double R[ORC_MAXL];
  orc_motion_bound(r, R);
#pragma omp parallel for schedule(dynamic, 4)
  for (int b = 0; b < B; ++b) {
    int hit = 0, und = 0, ev = 0;
    double th = -1.0, cm = INFINITY;
    for (int k = 0; k < H; ++k) {
      const double *xk = k == 0 ? x0 + (long)b * 2 * nj : x + ((long)b * H + (k - 1)) * 2 * nj;
      double tau, c;
      int e;
      const int v = orc_check_segment(r, nobs, obs, margin, R, xk, u + ((long)b * H + k) * nj, eta, max_evals, &tau, &c, &e);
      if (v == CHK_HIT && !hit) {
        hit = 1;
        th = (double)k * r->dt + tau;
      }
      und |= v == CHK_UNDECIDED;
      if (c < cm) cm = c;
      ev += e;
    }
    verdict[b] = hit ? CHK_HIT : (und ? CHK_UNDECIDED : CHK_CLEAR);
    t_hit[b] = th;
    cmin[b] = cm;
    evals[b] = ev;
  }
}
