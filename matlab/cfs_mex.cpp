// cfs_mex.cpp -- MEX gateway between the reference's MATLAB host code and libcfs_b200.so (include/cfs_b200.h).
//
//   [u, x_, cost_all, e_u_all, iters, status, qp_steps] = cfs_mex('solve', solver, grad, ROBOT, obs, sys_info [, noise])
//       (the first argument may be omitted: cfs_mex(solver, grad, ROBOT, obs, sys_info [, noise]))
//     solver   'CFS' | 'PSGCFS'                       (Lib/CFS_FANUC.m / Lib/PSGCFS_FANUC.m)
//     grad     'num_jac' | 'derivest'                 (Lib/functions/num_jac.m / DERIVESTsuite derivest.m on dist_link_*)
//     ROBOT    'M16iB' | 'M200i' | '2L'               (CFS_FANUC.m:49-54)
//     obs      cell of structs with fields l (3x2), D, epsilon                    (main_FANUC.m:56-60)
//     sys_info struct exactly as the mains build it                              (main_FANUC.m:106-127)
//              batched use: sys_info.xR (nstate x B), .ff (n x B), .caug (1 x B), .x_ (nstate*H x B)
//     noise    n x MAX_O_ITER x B normrnd(0,0.1) draws (PSGCFS_FANUC.m:109); REQUIRED for PSGCFS
//
//   [routes, route_len, n_nodes, fail, rnd_used, nodes, parent, total_dis] =
//       cfs_mex('rrt', ROBOT, SOLVER, obs, sys_info, goal, region_g, region_s, sample_off, rnd [, bi, max_iter])
//     RRT_FANUC.find_route (Lib/RRT_FANUC.m:63-207) for S = size(rnd,2) seeds at once (the parfor of
//     Lib/functions/s_Parallel_rrt.m:16-25).  SOLVER 'RRT' | 'RRT*'; sys_info.{x0, goal_th, ratial, nstate, robot};
//     rnd (nrnd x S): the uniform numbers of every seed, drawn in MATLAB (rand(nrnd,S)) and consumed in the reference's
//     order (pp = rand; rand(nstate,1) when pp < bi: RRT_FANUC.m:108,111).  routes: nstate x (max_iter+2) x S.
//
//   [u, x_, cost_all, e_u_all, iters, status] = cfs_mex('routes', ROBOT, obs, sys_info, routes, route_len, Q, Rblk, r_scale)
//     the CFS stage of RRTstar_CFS.m:96-195 for B routes (nstate x W x B, the first route_len(b) columns valid):
//     cubicpolytraj resampling to sys_info.H + 1 points, cost set-up from its blocks (Q 2nj x 2nj, Rblk nj x nj, R*r_scale),
//     CFS_FANUC.optimizer.  sys_info.{H, njoint, robot, lim, MAX_input, epsilon_O, MAX_O_ITER}.
//
//   [u, x_, cost_all, e_u_all, iters, status, verdict, t_hit, cmin, rounds_used, margin_off] =
//       cfs_mex('solve_checked', solver, grad, ROBOT, obs, sys_info [, noise [, eta, rounds, gain]])
//     'solve' followed by a continuous collision check of every trajectory and up to `rounds` re-solves of the HIT ones with
//     raised per-waypoint margins (extension; include/cfs_b200.h cfs_solve_checked).  solver 'CFS' | 'PSGCFS'; noise may be [];
//     eta = 1e-3, rounds = 4, gain = 2 by default.  verdict (1 x B int32: 0 clear, 1 hit, 2 undecided), t_hit, cmin (1 x B),
//     rounds_used (1 x B int32, 0 = the first solve), margin_off (H*nobs x B: reshape(margin_off(:, b), H, nobs) are the
//     offsets the returned solution of problem b was solved with).
//
//   [verdict, s_hit, cmin, evals] = cfs_mex('check', ROBOT, obs, sys_info, 'edges', A, B [, eta, margin_is_D])
//   [verdict, t_hit, cmin, evals] = cfs_mex('check', ROBOT, obs, sys_info, 'trajectory', x0, x_, u [, eta, margin_is_D])
//     continuous collision checks (extension; include/cfs_b200.h cfs_check_edges / cfs_check_trajectories): the edges
//     A(:,i) -> B(:,i) (njoint x N), or the solved trajectories x0 (nstate x B), x_ (nstate*H x B), u (njoint*H x B) between
//     their waypoints.  sys_info.robot and sys_info.njoint (or, for the RRT stage's sys_info, nstate).  eta = 1e-3 and
//     margin_is_D = 1 (obs{j}.D; 0: obs{j}.epsilon) by default.  verdict: 0 clear, 1 hit, 2 undecided (1 x N int32).
//
//   cfs_mex('device', id)   bind this MATLAB process to GPU `id` (call before anything else; parfor workers:
//                           cfs_mex('device', mod(labindex - 1, gpuDeviceCount)), see matlab/s_Parallel_rrt.m).
//                           Default: environment variable CFS_DEVICE, else 0.
//
// 'solve', 'solve_checked' and 'routes' read the optional sys_info.qlim (njoint x 2 = [min max] per joint): joint position limits of the
// CFS / PSGCFS solve (extension, include/cfs_b200.h cfs_set_joint_limits); a call without it solves without limits.
//
// Robot, obstacles and cost are cached by content hash: the Cholesky factor + Gram operator of cfs_set_cost (3.9 ms at
// n = 250) are rebuilt only when QQ / lim / MAX_input / H / robot really change between calls.
// Build (on a machine with MATLAB; this container has no mex.h, so the file is shipped as source and compiled against
// tests/mex_stub/mex.h by the test-suite):
//   mex -I<repo>/include cfs_mex.cpp -L<repo>/motionplanning_5d_m_b200 -lcfs_b200
// Export CUDA_DEVICE_MAX_CONNECTIONS=32 before starting MATLAB when more than 8 contexts (workers) share one GPU.
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "cfs_b200.h"
#include "mex.h"

static cfs_ctx *g_ctx = nullptr;
static int g_device = -1;
static uint64_t g_hash_robot = 0, g_hash_obs = 0, g_hash_cost = 0;

static void at_exit() {
  if (g_ctx) cfs_destroy(g_ctx);
  g_ctx = nullptr;
  g_hash_robot = g_hash_obs = g_hash_cost = 0;
}

static void check(int rc, const char *what) {
  if (rc != 0) mexErrMsgIdAndTxt("cfs:cuda", "%s failed (%d): %s", what, rc, cfs_last_error(g_ctx));
}

static uint64_t fnv(const void *p, size_t bytes, uint64_t h = 1469598103934665603ULL) {
  const unsigned char *c = static_cast<const unsigned char *>(p);
  for (size_t i = 0; i < bytes; ++i) h = (h ^ c[i]) * 1099511628211ULL;
  return h;
}

static const mxArray *field(const mxArray *s, const char *name, bool required = true) {
  if (!s || !mxIsStruct(s)) mexErrMsgIdAndTxt("cfs:arg", "expected a struct holding field '%s'", name);
  const mxArray *f = mxGetField(s, 0, name);
  if (!f && required) mexErrMsgIdAndTxt("cfs:arg", "missing field '%s'", name);
  return f;
}

// a real double array with exactly `count` elements (0 = any non-empty)
static const double *dbl(const mxArray *a, size_t count, const char *what) {
  if (!a || !mxIsDouble(a) || mxIsEmpty(a)) mexErrMsgIdAndTxt("cfs:arg", "%s must be a non-empty real double array", what);
  if (count && mxGetNumberOfElements(a) != count)
    mexErrMsgIdAndTxt("cfs:arg", "%s has %d elements, expected %d", what, (int)mxGetNumberOfElements(a), (int)count);
  return mxGetPr(a);
}

static double scalar(const mxArray *a, const char *what) { return dbl(a, 1, what)[0]; }

static std::string str(const mxArray *a) {
  char buf[64];
  if (!a || !mxIsChar(a) || mxGetString(a, buf, sizeof(buf))) mexErrMsgIdAndTxt("cfs:arg", "expected a short char array");
  return buf;
}

static int robot_kind(const std::string &name) {
  if (name == "M16iB") return CFS_ROBOT_M16IB;
  if (name == "M200i") return CFS_ROBOT_M200I;
  if (name == "2L") return CFS_ROBOT_2L;
  mexErrMsgIdAndTxt("cfs:arg", "unknown ROBOT '%s' (M16iB | M200i | 2L)", name.c_str());
  return -1;
}

static void ensure_ctx() {
  if (g_ctx) return;
  if (g_device < 0) {
    const char *env = std::getenv("CFS_DEVICE");
    g_device = env ? std::atoi(env) : 0;
  }
  cfs_ctx *c = nullptr;
  if (cfs_create(&c, g_device) != 0) mexErrMsgIdAndTxt("cfs:cuda", "%s", cfs_last_error(nullptr));  // no CPU fallback
  g_ctx = c;
  mexAtExit(at_exit);
}

// robotproperty2.m -> cfs_set_robot (cached)
static void bind_robot(const std::string &robot_name, const mxArray *rb, int nj) {
  const int kind = robot_kind(robot_name);
  const mxArray *DH = field(rb, "DH"), *cap = field(rb, "cap");
  const size_t dh_rows = mxGetM(DH);
  if (nj < 2 || nj > 6 || dh_rows < (size_t)nj) mexErrMsgIdAndTxt("cfs:arg", "njoint = %d with a %d-row DH table", nj, (int)dh_rows);
  dbl(DH, dh_rows * 4, "robot.DH");
  if (!mxIsCell(cap) || mxGetNumberOfElements(cap) < (size_t)nj) mexErrMsgIdAndTxt("cfs:arg", "robot.cap must be a cell with >= njoint entries");
  std::vector<double> cap_p(6 * nj);
  for (int i = 0; i < nj; ++i) {
    const mxArray *ci = mxGetCell(cap, i);
    if (!ci || !mxIsStruct(ci)) mexErrMsgIdAndTxt("cfs:arg", "robot.cap{%d} must be a struct with field p", i + 1);
    std::memcpy(&cap_p[6 * i], dbl(field(ci, "p"), 6, "robot.cap{i}.p (3x2)"), 6 * sizeof(double));
  }
  const mxArray *T = mxGetField(rb, 0, "T");
  if (kind == CFS_ROBOT_2L) dbl(T, 9, "robot.T (3x3)");
  const double dt = scalar(field(rb, "delta_t"), "robot.delta_t");
  const double *base = dbl(field(rb, "base"), 3, "robot.base");
  uint64_t h = fnv(&kind, sizeof(kind));
  h = fnv(&nj, sizeof(nj), h);
  h = fnv(mxGetPr(DH), sizeof(double) * dh_rows * 4, h);
  h = fnv(base, 3 * sizeof(double), h);
  h = fnv(cap_p.data(), cap_p.size() * sizeof(double), h);
  h = fnv(&dt, sizeof(dt), h);
  if (T && kind == CFS_ROBOT_2L) h = fnv(mxGetPr(T), 9 * sizeof(double), h);
  if (h == g_hash_robot) return;
  check(cfs_set_robot(g_ctx, kind, mxGetPr(DH), (int)dh_rows, base, cap_p.data(), nj, (T && kind == CFS_ROBOT_2L) ? mxGetPr(T) : nullptr, dt),
        "cfs_set_robot");
  g_hash_robot = h;
  g_hash_cost = 0;  // n depends on the robot
}

// obs{j}.{l, D, epsilon} (main_FANUC.m:56-60) -> cfs_set_obstacles (cached)
static void bind_obstacles(const mxArray *obs) {
  if (!obs || !mxIsCell(obs)) mexErrMsgIdAndTxt("cfs:arg", "obs must be a cell array of structs");
  const int nobs = (int)mxGetNumberOfElements(obs);
  std::vector<double> seg(6 * (nobs > 0 ? nobs : 1)), D(nobs > 0 ? nobs : 1), eps(nobs > 0 ? nobs : 1);
  std::vector<int> kind(nobs > 0 ? nobs : 1, CFS_OBS_CAPSULE);
  for (int j = 0; j < nobs; ++j) {
    const mxArray *o = mxGetCell(obs, j);
    if (!o || !mxIsStruct(o)) mexErrMsgIdAndTxt("cfs:arg", "obs{%d} must be a struct", j + 1);
    const mxArray *shape = mxGetField(o, 0, "shape");  // 'cylinder' (RRTstar_CFS.m:41) or, as an extension, 'box': l = [min max]
    if (shape && mxIsChar(shape) && str(shape) == "box") kind[j] = CFS_OBS_BOX;
    std::memcpy(&seg[6 * j], dbl(field(o, "l"), 6, "obs{j}.l (3x2)"), 6 * sizeof(double));
    D[j] = scalar(field(o, "D"), "obs{j}.D");
    const mxArray *e = field(o, "epsilon", false);
    eps[j] = e ? scalar(e, "obs{j}.epsilon") : D[j];
  }
  uint64_t h = fnv(&nobs, sizeof(nobs));
  h = fnv(seg.data(), sizeof(double) * 6 * nobs, h);
  h = fnv(D.data(), sizeof(double) * nobs, h);
  h = fnv(eps.data(), sizeof(double) * nobs, h);
  h = fnv(kind.data(), sizeof(int) * nobs, h);
  if (h == g_hash_obs) return;
  check(cfs_set_obstacles_ex(g_ctx, seg.data(), kind.data(), D.data(), eps.data(), nobs), "cfs_set_obstacles_ex");
  g_hash_obs = h;
}

static void out_int(mxArray *&dst, const std::vector<int> &v) {
  dst = mxCreateNumericMatrix(1, v.size(), mxINT32_CLASS, mxREAL);
  if (!v.empty()) std::memcpy(mxGetData(dst), v.data(), sizeof(int) * v.size());
}

// ---- 'solve' ------------------------------------------------------------------------------------------------------------------
// joint position limits (extension, cfs_set_joint_limits) from the optional sys_info.qlim = [min max] per joint (njoint x 2),
// set or cleared by every command that solves (si == nullptr: cleared): the cached context never keeps the limits of an
// earlier call
static void bind_qlim(const mxArray *si, int nj) {
  const mxArray *ql = si ? field(si, "qlim", false) : nullptr;
  if (ql && (mxGetM(ql) != (size_t)nj || mxGetN(ql) != 2)) mexErrMsgIdAndTxt("cfs:arg", "sys_info.qlim must be njoint x 2 ([min max])");
  const double *qlp = ql ? dbl(ql, 2 * (size_t)nj, "sys_info.qlim (njoint x 2)") : nullptr;
  check(cfs_set_joint_limits(g_ctx, qlp, qlp ? qlp + nj : nullptr), "cfs_set_joint_limits");
}

// checked: the 'solve_checked' command (cfs_solve_checked), prhs[6..8] = eta, rounds, gain (optional)
static void cmd_solve(int nlhs, mxArray *plhs[], int nrhs, const mxArray *prhs[], bool checked = false) {
  if (nrhs < 5)
    mexErrMsgIdAndTxt("cfs:arg", checked ? "usage: cfs_mex('solve_checked', solver, grad, ROBOT, obs, sys_info [, noise [, eta, rounds, gain]])"
                                         : "usage: cfs_mex('solve', solver, grad, ROBOT, obs, sys_info [, noise | uu])");
  const std::string solver = str(prhs[0]), grad = str(prhs[1]), robot_name = str(prhs[2]);
  if (checked && solver == "CHOMP") mexErrMsgIdAndTxt("cfs:arg", "solve_checked: solver '%s' (CFS | PSGCFS)", solver.c_str());
  if (solver != "CFS" && solver != "PSGCFS" && solver != "CHOMP")
    mexErrMsgIdAndTxt("cfs:arg", "solver '%s' (CFS | PSGCFS | CHOMP)", solver.c_str());
  const bool chomp = solver == "CHOMP";
  if (grad != "num_jac" && grad != "derivest") mexErrMsgIdAndTxt("cfs:arg", "grad '%s' (num_jac | derivest)", grad.c_str());
  const mxArray *obs = prhs[3], *si = prhs[4];
  const int H = (int)scalar(field(si, "H"), "sys_info.H"), nj = (int)scalar(field(si, "njoint"), "sys_info.njoint");
  if (H < 1) mexErrMsgIdAndTxt("cfs:arg", "sys_info.H = %d", H);
  const size_t n = (size_t)H * nj;
  ensure_ctx();
  bind_robot(robot_name, field(si, "robot"), nj);
  bind_obstacles(obs);
  // ---- cost (main_FANUC.m:106-127); PSGCFS projects without bounds (PSGCFS_FANUC.m:120) -----------------------------
  const bool psg = solver == "PSGCFS";
  const mxArray *lim = field(si, "lim", false), *mi = field(si, "MAX_input", false);
  const double *QQ = dbl(field(si, "QQ"), n * n, "sys_info.QQ (n x n)");
  const double *limp = lim ? dbl(lim, nj, "sys_info.lim (njoint)") : nullptr;
  const double *mip = (mi && !psg) ? dbl(mi, n, "sys_info.MAX_input (n)") : nullptr;
  uint64_t h = fnv(&H, sizeof(H));
  h = fnv(QQ, sizeof(double) * n * n, h);
  if (limp) h = fnv(limp, sizeof(double) * nj, h);
  if (mip) h = fnv(mip, sizeof(double) * n, h);
  h = fnv(&psg, sizeof(psg), h) ^ 0x51ULL;
  if (h != g_hash_cost) {
    check(cfs_set_cost(g_ctx, H, QQ, limp, mip), "cfs_set_cost");
    g_hash_cost = h;
  }
  bind_qlim(chomp ? nullptr : si, nj);  // CHOMP does not read the limits
  // ---- the batch ----------------------------------------------------------------------------------------------------
  const mxArray *xR = field(si, "xR"), *ff = field(si, "ff"), *caug = field(si, "caug"), *xref = field(si, "x_");
  const size_t B = mxGetNumberOfElements(caug);
  if (B == 0) mexErrMsgIdAndTxt("cfs:arg", "sys_info.caug is empty: no problem to solve");
  dbl(ff, n * B, "sys_info.ff (n x B)");
  dbl(xref, 2 * n * B, "sys_info.x_ (nstate*H x B)");
  dbl(xR, 0, "sys_info.xR");
  const int K = (int)scalar(field(si, "MAX_O_ITER"), "sys_info.MAX_O_ITER");
  if (K < 0) mexErrMsgIdAndTxt("cfs:arg", "sys_info.MAX_O_ITER = %d", K);
  const size_t xr_rows = mxGetM(xR), xr_cols = mxGetN(xR);
  if (xr_rows < (size_t)2 * nj || xr_cols < B || xr_cols % B != 0)
    mexErrMsgIdAndTxt("cfs:arg", "sys_info.xR is %d x %d, expected nstate x B (or nstate x (H+1) for B = 1)", (int)xr_rows, (int)xr_cols);
  std::vector<double> x0((size_t)2 * nj * B);
  const size_t ldxr = xr_rows * (xr_cols / B);  // sys_info.xR may carry later roll-out columns (B = 1)
  for (size_t b = 0; b < B; ++b) std::memcpy(&x0[(size_t)2 * nj * b], mxGetPr(xR) + ldxr * b, 2 * nj * sizeof(double));
  const double *noise = nullptr;
  if (chomp) {  // CHOMP_FANUC(obs, sys_info, uu, ROBOT): the initial controls (Lib/CHOMP_FANUC.m:34,48)
    if (nrhs < 6 || !prhs[5] || mxIsEmpty(prhs[5])) mexErrMsgIdAndTxt("cfs:arg", "CHOMP needs the initial controls uu (n x B)");
    noise = dbl(prhs[5], n * B, "uu (n x B)");
  } else if (nrhs > 5 && prhs[5] && !mxIsEmpty(prhs[5])) {
    noise = dbl(prhs[5], n * (size_t)K * B, "noise (n x MAX_O_ITER x B)");
  }
  if (psg && !noise && K > 0)
    mexErrMsgIdAndTxt("cfs:arg", "PSGCFS needs the normrnd(0,0.1,[nn,1]) draws of every outer iteration (PSGCFS_FANUC.m:109) as "
                                 "noise (n x MAX_O_ITER x B); matlab/PSGCFS_FANUC.m draws them");
  const mxArray *alpha = field(si, "alpha", false);
  plhs[0] = mxCreateDoubleMatrix(n, B, mxREAL);
  mxArray *x = mxCreateDoubleMatrix(2 * n, B, mxREAL), *cost = mxCreateDoubleMatrix(K > 0 ? K : 1, B, mxREAL),
          *eu = mxCreateDoubleMatrix(K > 0 ? K : 1, B, mxREAL);
  mxArray *it = mxCreateNumericMatrix(1, B, mxINT32_CLASS, mxREAL), *st = mxCreateNumericMatrix(1, B, mxINT32_CLASS, mxREAL);
  if (checked) {
    auto opt = [&](int i, double def, const char *what) {
      return (nrhs > i && prhs[i] && !mxIsEmpty(prhs[i])) ? scalar(prhs[i], what) : def;
    };
    const double eta = opt(6, 1e-3, "eta"), gain = opt(8, 2.0, "gain");
    const int rounds = (int)opt(7, 4.0, "rounds");
    const size_t OH = mxGetNumberOfElements(obs) * (size_t)H;
    mxArray *vd = mxCreateNumericMatrix(1, B, mxINT32_CLASS, mxREAL), *th = mxCreateDoubleMatrix(1, B, mxREAL),
            *cm = mxCreateDoubleMatrix(1, B, mxREAL), *ru = mxCreateNumericMatrix(1, B, mxINT32_CLASS, mxREAL),
            *mo = mxCreateDoubleMatrix(OH, B, mxREAL);
    check(cfs_solve_checked(g_ctx, (int)B, psg ? CFS_SOLVER_PSGCFS : CFS_SOLVER_CFS, grad == "derivest" ? CFS_GRAD_DERIVEST : CFS_GRAD_NUMJAC,
                            x0.data(), mxGetPr(ff), mxGetPr(caug), mxGetPr(xref), noise, scalar(field(si, "epsilon_O"), "sys_info.epsilon_O"),
                            K, alpha ? scalar(alpha, "sys_info.alpha") : 0.0, eta, 4096, rounds, gain, mxGetPr(plhs[0]), mxGetPr(x),
                            mxGetPr(cost), mxGetPr(eu), (int *)mxGetData(it), (int *)mxGetData(st), (int *)mxGetData(vd), mxGetPr(th),
                            mxGetPr(cm), (int *)mxGetData(ru), OH ? mxGetPr(mo) : nullptr),
          "cfs_solve_checked");
    mxArray *outs[11] = {plhs[0], x, cost, eu, it, st, vd, th, cm, ru, mo};
    for (int k = 1; k < 11 && k < nlhs; ++k) plhs[k] = outs[k];
    return;
  }
  if (chomp) {
    if (!alpha) mexErrMsgIdAndTxt("cfs:arg", "CHOMP needs sys_info.alpha");
    check(cfs_chomp_batch(g_ctx, (int)B, x0.data(), mxGetPr(ff), mxGetPr(caug), mxGetPr(xref), noise, scalar(alpha, "sys_info.alpha"), K,
                          mxGetPr(plhs[0]), mxGetPr(x), mxGetPr(cost), mxGetPr(eu), (int *)mxGetData(it), (int *)mxGetData(st)),
          "cfs_chomp_batch");
  } else
  check(cfs_solve_batch(g_ctx, (int)B, psg ? CFS_SOLVER_PSGCFS : CFS_SOLVER_CFS, grad == "derivest" ? CFS_GRAD_DERIVEST : CFS_GRAD_NUMJAC,
                        x0.data(), mxGetPr(ff), mxGetPr(caug), mxGetPr(xref), noise, scalar(field(si, "epsilon_O"), "sys_info.epsilon_O"), K,
                        alpha ? scalar(alpha, "sys_info.alpha") : 0.0, mxGetPr(plhs[0]), mxGetPr(x), mxGetPr(cost), mxGetPr(eu),
                        (int *)mxGetData(it), (int *)mxGetData(st)), "cfs_solve_batch");
  if (nlhs > 1) plhs[1] = x;
  if (nlhs > 2) plhs[2] = cost;
  if (nlhs > 3) plhs[3] = eu;
  if (nlhs > 4) plhs[4] = it;
  if (nlhs > 5) plhs[5] = st;
  if (nlhs > 6) {
    cfs_stats s;
    cfs_get_stats(g_ctx, &s);
    plhs[6] = mxCreateDoubleScalar((double)s.qp_steps);
  }
}

// ---- 'rrt' --------------------------------------------------------------------------------------------------------------------
static void cmd_rrt(int nlhs, mxArray *plhs[], int nrhs, const mxArray *prhs[]) {
  if (nrhs < 9)
    mexErrMsgIdAndTxt("cfs:arg", "usage: cfs_mex('rrt', ROBOT, SOLVER, obs, sys_info, goal, region_g, region_s, sample_off, rnd [, bi, max_iter])");
  const std::string robot_name = str(prhs[0]), solver = str(prhs[1]);
  if (solver != "RRT" && solver != "RRT*") mexErrMsgIdAndTxt("cfs:arg", "SOLVER '%s' (RRT | RRT*)", solver.c_str());
  const mxArray *obs = prhs[2], *si = prhs[3];
  const int nj = (int)scalar(field(si, "nstate"), "sys_info.nstate");
  ensure_ctx();
  bind_robot(robot_name, field(si, "robot"), nj);
  bind_obstacles(obs);
  const double *goal = dbl(prhs[4], nj, "goal"), *rg = dbl(prhs[5], nj, "region_g"), *rs = dbl(prhs[6], nj, "region_s"),
               *off = dbl(prhs[7], nj, "sample_off");
  const double *x0 = dbl(field(si, "x0"), nj, "sys_info.x0"), *gth = dbl(field(si, "goal_th"), nj, "sys_info.goal_th"),
               *rat = dbl(field(si, "ratial"), nj, "sys_info.ratial");
  const mxArray *rnd = prhs[8];
  dbl(rnd, 0, "rnd (nrnd x S)");
  const int nrnd = (int)mxGetM(rnd), S = (int)mxGetN(rnd);
  if (nrnd < 1 || S < 1) mexErrMsgIdAndTxt("cfs:arg", "rnd must be nrnd x S");
  const double bi = nrhs > 9 ? scalar(prhs[9], "bi") : 0.5;                       // RRT_FANUC.m:38
  const int max_iter = nrhs > 10 ? (int)scalar(prhs[10], "max_iter") : 400;      // RRT_FANUC.m:37
  if (max_iter < 1) mexErrMsgIdAndTxt("cfs:arg", "max_iter = %d", max_iter);
  const int cap = max_iter + 2;
  std::vector<double> X0((size_t)nj * S), G((size_t)nj * S), GT((size_t)nj * S);
  for (int s = 0; s < S; ++s) {
    std::memcpy(&X0[(size_t)nj * s], x0, nj * sizeof(double));
    std::memcpy(&G[(size_t)nj * s], goal, nj * sizeof(double));
    std::memcpy(&GT[(size_t)nj * s], gth, nj * sizeof(double));
  }
  plhs[0] = mxCreateDoubleMatrix((size_t)nj * cap, S, mxREAL);  // nstate x (max_iter+2) x S, reshape in MATLAB
  std::vector<int> len(S), nn(S), fl(S), used(S), par((size_t)cap * S);
  mxArray *nodes = mxCreateDoubleMatrix((size_t)nj * cap, S, mxREAL), *tot = mxCreateDoubleMatrix(cap, S, mxREAL);
  check(cfs_rrt_find_routes(g_ctx, S, solver == "RRT*" ? 1 : 0, X0.data(), G.data(), GT.data(), rg, rs, off, rat, bi, max_iter,
                            mxGetPr(rnd), nrnd, mxGetPr(plhs[0]), len.data(), nn.data(), fl.data(), used.data(), mxGetPr(nodes),
                            par.data(), mxGetPr(tot), nullptr), "cfs_rrt_find_routes");
  if (nlhs > 1) out_int(plhs[1], len);
  if (nlhs > 2) out_int(plhs[2], nn);
  if (nlhs > 3) out_int(plhs[3], fl);
  if (nlhs > 4) out_int(plhs[4], used);
  if (nlhs > 5) plhs[5] = nodes;
  if (nlhs > 6) {
    plhs[6] = mxCreateNumericMatrix(cap, S, mxINT32_CLASS, mxREAL);
    std::memcpy(mxGetData(plhs[6]), par.data(), sizeof(int) * par.size());
  }
  if (nlhs > 7) plhs[7] = tot;
}

// ---- 'routes' -----------------------------------------------------------------------------------------------------------------
static void cmd_routes(int nlhs, mxArray *plhs[], int nrhs, const mxArray *prhs[]) {
  if (nrhs < 8) mexErrMsgIdAndTxt("cfs:arg", "usage: cfs_mex('routes', ROBOT, obs, sys_info, routes, route_len, Q, Rblk, r_scale)");
  const std::string robot_name = str(prhs[0]);
  const mxArray *obs = prhs[1], *si = prhs[2], *routes = prhs[3], *rl = prhs[4];
  const int H = (int)scalar(field(si, "H"), "sys_info.H"), nj = (int)scalar(field(si, "njoint"), "sys_info.njoint");
  if (H < 1) mexErrMsgIdAndTxt("cfs:arg", "sys_info.H = %d", H);
  const size_t n = (size_t)H * nj;
  const size_t B = mxGetNumberOfElements(rl);
  dbl(rl, 0, "route_len (1 x B)");
  dbl(routes, 0, "routes (nstate x W x B)");
  const size_t tot = mxGetNumberOfElements(routes);
  if (tot % ((size_t)nj * B) != 0) mexErrMsgIdAndTxt("cfs:arg", "routes has %d elements: not nstate x W x B with B = %d", (int)tot, (int)B);
  const int W = (int)(tot / ((size_t)nj * B));
  if (W < 2) mexErrMsgIdAndTxt("cfs:arg", "routes need at least two waypoints (W = %d)", W);
  std::vector<int> len(B);
  for (size_t b = 0; b < B; ++b) {
    const double v = mxGetPr(rl)[b];
    len[b] = v < 0 ? 0 : (v > W ? W : (int)v);
  }
  ensure_ctx();
  bind_robot(robot_name, field(si, "robot"), nj);
  bind_obstacles(obs);
  const double *Q = dbl(prhs[5], (size_t)4 * nj * nj, "Q (2nj x 2nj)"), *Rb = dbl(prhs[6], (size_t)nj * nj, "Rblk (nj x nj)");
  const double r_scale = scalar(prhs[7], "r_scale");
  const mxArray *lim = field(si, "lim", false), *mi = field(si, "MAX_input", false);
  const double *limp = lim ? dbl(lim, nj, "sys_info.lim") : nullptr, *mip = mi ? dbl(mi, n, "sys_info.MAX_input") : nullptr;
  uint64_t h = fnv(&H, sizeof(H));
  h = fnv(Q, sizeof(double) * 4 * nj * nj, h);
  h = fnv(Rb, sizeof(double) * nj * nj, h);
  h = fnv(&r_scale, sizeof(r_scale), h);
  if (limp) h = fnv(limp, sizeof(double) * nj, h);
  if (mip) h = fnv(mip, sizeof(double) * n, h);
  h ^= 0xb10cULL;
  if (h != g_hash_cost) {
    check(cfs_set_cost_blocks(g_ctx, H, Q, Rb, r_scale, 0.1, 10000.0, limp, mip), "cfs_set_cost_blocks");  // RRTstar_CFS.m:139-150
    g_hash_cost = h;
  }
  bind_qlim(si, nj);
  const int K = (int)scalar(field(si, "MAX_O_ITER"), "sys_info.MAX_O_ITER");
  plhs[0] = mxCreateDoubleMatrix(n, B, mxREAL);
  mxArray *x = mxCreateDoubleMatrix(2 * n, B, mxREAL), *cost = mxCreateDoubleMatrix(K > 0 ? K : 1, B, mxREAL),
          *eu = mxCreateDoubleMatrix(K > 0 ? K : 1, B, mxREAL);
  mxArray *it = mxCreateNumericMatrix(1, B, mxINT32_CLASS, mxREAL), *st = mxCreateNumericMatrix(1, B, mxINT32_CLASS, mxREAL);
  check(cfs_solve_routes_var(g_ctx, (int)B, W, len.data(), CFS_SOLVER_CFS, CFS_GRAD_NUMJAC, mxGetPr(routes), nullptr,
                             scalar(field(si, "epsilon_O"), "sys_info.epsilon_O"), K, 0.0, mxGetPr(plhs[0]), mxGetPr(x), mxGetPr(cost),
                             mxGetPr(eu), (int *)mxGetData(it), (int *)mxGetData(st)), "cfs_solve_routes_var");
  if (nlhs > 1) plhs[1] = x;
  if (nlhs > 2) plhs[2] = cost;
  if (nlhs > 3) plhs[3] = eu;
  if (nlhs > 4) plhs[4] = it;
  if (nlhs > 5) plhs[5] = st;
}

// ---- 'check' ------------------------------------------------------------------------------------------------------------------
static void cmd_check(int nlhs, mxArray *plhs[], int nrhs, const mxArray *prhs[]) {
  if (nrhs < 6)
    mexErrMsgIdAndTxt("cfs:arg", "usage: cfs_mex('check', ROBOT, obs, sys_info, 'edges', A, B [, eta, margin_is_D]) or "
                                 "cfs_mex('check', ROBOT, obs, sys_info, 'trajectory', x0, x_, u [, eta, margin_is_D])");
  const std::string robot_name = str(prhs[0]), what = str(prhs[3]);
  const mxArray *obs = prhs[1], *si = prhs[2];
  if (what != "edges" && what != "trajectory") mexErrMsgIdAndTxt("cfs:arg", "check '%s' (edges | trajectory)", what.c_str());
  const bool edges = what == "edges";
  if (!edges && nrhs < 7) mexErrMsgIdAndTxt("cfs:arg", "usage: cfs_mex('check', ROBOT, obs, sys_info, 'trajectory', x0, x_, u [, eta, margin_is_D])");
  const mxArray *njf = field(si, "njoint", false);
  const int nj = (int)scalar(njf ? njf : field(si, "nstate"), "sys_info.njoint");
  const int nopt = edges ? 6 : 7;
  const double eta = nrhs > nopt ? scalar(prhs[nopt], "eta") : 1e-3;
  const int margin_is_D = nrhs > nopt + 1 ? (scalar(prhs[nopt + 1], "margin_is_D") != 0.0) : 1;
  ensure_ctx();
  bind_robot(robot_name, field(si, "robot"), nj);
  bind_obstacles(obs);
  const size_t N = mxGetN(prhs[4]);
  std::vector<int> verdict(N), evals(N);
  mxArray *where = mxCreateDoubleMatrix(1, N, mxREAL), *cmin = mxCreateDoubleMatrix(1, N, mxREAL);
  if (edges) {
    const double *A = dbl(prhs[4], (size_t)nj * N, "A (njoint x N)"), *B = dbl(prhs[5], (size_t)nj * N, "B (njoint x N)");
    check(cfs_check_edges(g_ctx, (int)N, A, B, eta, margin_is_D, 4096, verdict.data(), mxGetPr(where), mxGetPr(cmin), evals.data()),
          "cfs_check_edges");
  } else {
    const double *x0 = dbl(prhs[4], (size_t)2 * nj * N, "x0 (nstate x B)");
    const double *u = dbl(prhs[6], 0, "u (njoint*H x B)");
    const size_t nu = mxGetNumberOfElements(prhs[6]);
    if (N == 0 || nu % ((size_t)nj * N) != 0) mexErrMsgIdAndTxt("cfs:arg", "u has %d elements: not njoint*H x B with B = %d", (int)nu, (int)N);
    const int H = (int)(nu / ((size_t)nj * N));
    const double *x = dbl(prhs[5], (size_t)2 * nj * H * N, "x_ (nstate*H x B)");
    check(cfs_check_trajectories(g_ctx, (int)N, H, x0, x, u, eta, margin_is_D, 4096, verdict.data(), mxGetPr(where), mxGetPr(cmin),
                                 evals.data()), "cfs_check_trajectories");
  }
  out_int(plhs[0], verdict);
  if (nlhs > 1) plhs[1] = where;
  if (nlhs > 2) plhs[2] = cmin;
  if (nlhs > 3) out_int(plhs[3], evals);
}

void mexFunction(int nlhs, mxArray *plhs[], int nrhs, const mxArray *prhs[]) {
  if (nrhs < 1) mexErrMsgIdAndTxt("cfs:arg", "usage: cfs_mex(command, ...); commands: solve, solve_checked, rrt, routes, check, device");
  const std::string cmd = str(prhs[0]);
  if (cmd == "device") {
    if (nrhs < 2) mexErrMsgIdAndTxt("cfs:arg", "usage: cfs_mex('device', id)");
    const int id = (int)scalar(prhs[1], "device id");
    if (g_ctx && id != g_device) at_exit();  // re-bind: the next call creates the context on the new device
    g_device = id;
    return;
  }
  if (cmd == "solve") return cmd_solve(nlhs, plhs, nrhs - 1, prhs + 1);
  if (cmd == "rrt") return cmd_rrt(nlhs, plhs, nrhs - 1, prhs + 1);
  if (cmd == "routes") return cmd_routes(nlhs, plhs, nrhs - 1, prhs + 1);
  if (cmd == "check") return cmd_check(nlhs, plhs, nrhs - 1, prhs + 1);
  if (cmd == "solve_checked") return cmd_solve(nlhs, plhs, nrhs - 1, prhs + 1, true);
  if (cmd == "CFS" || cmd == "PSGCFS" || cmd == "CHOMP") return cmd_solve(nlhs, plhs, nrhs, prhs);  // short calling form
  mexErrMsgIdAndTxt("cfs:arg", "unknown command '%s' (solve | solve_checked | rrt | routes | check | device)", cmd.c_str());
}
