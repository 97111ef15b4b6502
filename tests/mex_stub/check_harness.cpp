// check_harness.cpp -- the stub harness (harness.cpp: mex.h stand-in, argument builders, the existing mexh_* entries) plus an
// entry point for the gateway's 'check' command.  Test infrastructure only; tests/test_mex_check.py compiles it together with
// matlab/cfs_mex.cpp into a library of its own.
#include "harness.cpp"

// [verdict, s_hit | t_hit, cmin, evals] = cfs_mex('check', ROBOT, obs, sys_info, what, a, b [, c], eta, margin_is_D)
//   what = "edges": a = A, b = B (nj x N);  what = "trajectory": a = x0 (2nj x N), b = x_ (2njH x N), c = u (njH x N)
extern "C" int mexh_check(const char *robot_name, int nj, int dh_rows, const double *DH, const double *base, const double *cap_p,
                          const double *T, double dt, int nobs, const double *obs_l, const double *obs_D, const double *obs_eps,
                          const char *what, int N, int H, const double *a, const double *b, const double *c, double eta,
                          int margin_is_D, int *verdict, double *where, double *cmin, int *evals) {
  g_err[0] = 0;
  const bool edges = std::strcmp(what, "edges") == 0;
  mxArray *si = strct();
  const double njd = nj, mD = margin_is_D;
  si->fields["njoint"] = dbl(1, 1, &njd);
  si->fields["robot"] = robot_struct(nj, dh_rows, DH, base, cap_p, T, dt);
  std::vector<const mxArray *> prhs = {chr("check"), chr(robot_name), obs_cell(nobs, obs_l, obs_D, obs_eps), si, chr(what)};
  if (edges) {
    prhs.push_back(dbl(nj, N, a));
    prhs.push_back(dbl(nj, N, b));
  } else {
    prhs.push_back(dbl(2 * nj, N, a));
    prhs.push_back(dbl((size_t)2 * nj * H, N, b));
    prhs.push_back(dbl((size_t)nj * H, N, c));
  }
  prhs.push_back(dbl(1, 1, &eta));
  prhs.push_back(dbl(1, 1, &mD));
  mxArray *plhs[4] = {nullptr};
  int rc = 0;
  try {
    mexFunction(4, plhs, (int)prhs.size(), prhs.data());
    std::memcpy(verdict, plhs[0]->i32.data(), sizeof(int) * N);
    std::memcpy(where, plhs[1]->d.data(), sizeof(double) * N);
    std::memcpy(cmin, plhs[2]->d.data(), sizeof(double) * N);
    std::memcpy(evals, plhs[3]->i32.data(), sizeof(int) * N);
  } catch (const mex_error &e) {
    snprintf(g_err, sizeof(g_err), "%s: %s", e.id.c_str(), e.msg.c_str());
    rc = 1;
  }
  return finish(rc);
}

