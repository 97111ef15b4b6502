// limits_harness.cpp -- the stub harness (harness.cpp) plus an entry point for the gateway's 'solve' command with the optional
// sys_info.qlim.  Test infrastructure only; tests/test_mex_limits.py compiles it together with matlab/cfs_mex.cpp into a library
// of its own.
#include "harness.cpp"

// [u, x_, cost_all, e_u_all, iters, status] = cfs_mex('solve', 'CFS', 'num_jac', ROBOT, obs, sys_info) with sys_info.qlim = qlim
// (njoint x 2 column-major, [min max]) or without the field (qlim NULL).  All matrices column-major as MATLAB stores them.
extern "C" int mexh_solve_qlim(const char *robot_name, int nj, int H, int B, int dh_rows, const double *DH, const double *base,
                               const double *cap_p, double dt, int nobs, const double *obs_l, const double *obs_D,
                               const double *obs_eps, const double *QQ, const double *lim, const double *max_input,
                               const double *qlim, const double *xR, const double *ff, const double *caug, const double *xref,
                               double eps_outer, int max_outer, double *u, double *x, double *cost, double *eu, int *iters,
                               int *status) {
  const size_t n = (size_t)H * nj;
  g_err[0] = 0;
  mxArray *si = strct();
  const double Hd = H, njd = nj, Kd = max_outer;
  si->fields["H"] = dbl(1, 1, &Hd);
  si->fields["njoint"] = dbl(1, 1, &njd);
  si->fields["robot"] = robot_struct(nj, dh_rows, DH, base, cap_p, nullptr, dt);
  si->fields["QQ"] = dbl(n, n, QQ);
  if (lim) si->fields["lim"] = dbl(nj, 1, lim);
  if (max_input) si->fields["MAX_input"] = dbl(n, 1, max_input);
  if (qlim) si->fields["qlim"] = dbl(nj, 2, qlim);
  si->fields["xR"] = dbl(2 * nj, B, xR);
  si->fields["ff"] = dbl(n, B, ff);
  si->fields["caug"] = dbl(1, B, caug);
  si->fields["x_"] = dbl(2 * n, B, xref);
  si->fields["epsilon_O"] = dbl(1, 1, &eps_outer);
  si->fields["MAX_O_ITER"] = dbl(1, 1, &Kd);
  const mxArray *prhs[6] = {chr("solve"), chr("CFS"), chr("num_jac"), chr(robot_name), obs_cell(nobs, obs_l, obs_D, obs_eps), si};
  mxArray *plhs[6] = {nullptr};
  int rc = 0;
  try {
    mexFunction(6, plhs, 6, prhs);
    std::memcpy(u, plhs[0]->d.data(), sizeof(double) * n * B);
    std::memcpy(x, plhs[1]->d.data(), sizeof(double) * 2 * n * B);
    std::memcpy(cost, plhs[2]->d.data(), sizeof(double) * max_outer * B);
    std::memcpy(eu, plhs[3]->d.data(), sizeof(double) * max_outer * B);
    std::memcpy(iters, plhs[4]->i32.data(), sizeof(int) * B);
    std::memcpy(status, plhs[5]->i32.data(), sizeof(int) * B);
  } catch (const mex_error &e) {
    snprintf(g_err, sizeof(g_err), "%s: %s", e.id.c_str(), e.msg.c_str());
    rc = 1;
  }
  return finish(rc);
}
