/*
 * cfs_b200.h -- C ABI of libcfs_b200.so: the B200-native (sm_100a) Convex-Feasible-Set hot path.
 *
 * Drop-in boundary for JessicaLeu-code/MotionPlanning_5D_m.  The reference has no FFI layer of
 * its own; the boundary is the MATLAB class contract used by its mains
 *     self = CFS_FANUC(obs, sys_info, ROBOT); self = self.optimizer();     (main_FANUC.m:150-151,
 *     RRTstar_CFS.m:194-195, Lib/functions/s_Solver.m:33-36)
 * and every entry point below replaces the body of one reference function (cited per function).
 * A MEX gateway (matlab/cfs_mex.cpp) or any FFI (ctypes: motionplanning_5d_m_b200/_lib.py) binds
 * exactly these symbols.  See INTEGRATION.md.
 *
 * Conventions
 *   - all arrays are column-major FP64 exactly as MATLAB stores them; "n x B" means problem b
 *     occupies elements [n*b, n*(b+1)).
 *   - caller owns every host buffer; the library owns all device memory behind cfs_ctx.
 *   - return value: 0 = ok, <0 = CFS_E_* (message via cfs_last_error).  Per-problem outcomes go
 *     to status[] and never to the return code.
 *   - one cfs_ctx is bound to one CUDA device and one stream; it is not thread-safe, but any
 *     number of contexts/processes may coexist (MATLAB parfor workers: s_Parallel_rrt.m:16).
 *   - there is NO CPU fallback: every entry point fails with CFS_E_CUDA if no sm_100 device
 *     is usable.
 */
#ifndef CFS_B200_H
#define CFS_B200_H

#ifdef __cplusplus
extern "C" {
#endif

typedef struct cfs_ctx cfs_ctx;

/* robot_kind: selects the FK flavour / joint offset exactly as CFS_FANUC.m:49-54 selects dist_arm_all */
enum { CFS_ROBOT_M16IB = 0, /* Lib/M16iB/dist_arm_3D_Heu_2.m */
       CFS_ROBOT_M200I = 1, /* Lib/200i/dist_arm_3D_200i_2.m (joint 2 offset -pi/2, :11) */
       CFS_ROBOT_2L = 2 };  /* Lib/2L/dist_arm_2L.m + CapPos2.m */

enum { CFS_SOLVER_CFS = 0,     /* Lib/CFS_FANUC.m    */
       CFS_SOLVER_PSGCFS = 1 };/* Lib/PSGCFS_FANUC.m */

enum { CFS_GRAD_NUMJAC = 0,    /* Lib/functions/num_jac.m (class path, CFS_FANUC.m:118) */
       CFS_GRAD_DERIVEST = 1 };/* derivest on dist_link_*(linkid) (script path, M16iB/main_CFS.m:234-237) */

/* status[b] low byte */
enum { CFS_STATUS_CONVERGED = 0,  /* ||x_-x_old|| < epsilon_O                 (EVAL.m:64-67)  */
       CFS_STATUS_MAX_ITER = 1,   /* iter_O > MAX_O_ITER                      (EVAL.m:69-72)  */
       CFS_STATUS_INFEASIBLE = 2, /* QP infeasible: quadprog returns [] and the reference's rollout throws (CFS_FANUC.m:85-92) */
       CFS_STATUS_NUMERICAL = 3,
       CFS_STATUS_NO_ROUTE = 5 }; /* cfs_solve_routes_var: route_len < 2, i.e. the RRT seed failed (RRT_FANUC.m:201-205; routeL = 1000
                                     in Lib/functions/s_Parallel_rrt.m:11): nothing to smooth, u = 0 */
/* status[b] flag bits */
#define CFS_FLAG_TOUCH 0x100 /* the |dis|<1e-4 "axes touch" branch was taken at some evaluated configuration
                                (dist_arm_3D_Heu_2.m:22-24).  On M16iB the reference subtracts a 3x1 from a 6x1
                                there and throws; this library evaluates the 200i/dist_link form points(1:3). */

enum { CFS_E_ARG = -1, CFS_E_CUDA = -2, CFS_E_STATE = -3, CFS_E_NOMEM = -4, CFS_E_NUMERIC = -5 };

/* ---- context ------------------------------------------------------------------------------------------ */
int         cfs_create(cfs_ctx **out, int device_id);
void        cfs_destroy(cfs_ctx *ctx);
const char *cfs_last_error(const cfs_ctx *ctx); /* ctx may be NULL: returns the last creation error */
const char *cfs_version(void);
/* Run on a caller-owned CUDA stream (cudaStream_t passed as void*; e.g. torch.cuda.current_stream().cuda_stream) so that
 * the caller's events bracket the library's kernels.  NULL restores the context's own stream. */
int cfs_set_stream(cfs_ctx *ctx, void *cuda_stream);

/* Options: "fused" (default 1): solve CFS / num_jac batches with the persistent fused kernel (one CTA carries a problem
 * through all outer iterations); 0 = one gradient launch + one QP launch per outer iteration (the path PSGCFS and the
 * DERIVEST gradients always take).  "esc_steps" (default 48): dual active-set steps one QP may take in the fused
 * kernel's bulk tier before the problem is handed to its heavy tier (0 = never).  Scheduling knobs, none of which changes a
 * result: "lpt" (default 1): the fused solver pulls the problems longest-expected-first (a distance pre-pass over every
 * reference line orders them by the number of waypoints inside an obstacle margin); "bulk_grid" / "heavy_grid" (default 0 =
 * every resident slot / 48 CTAs): caps of the two tiers' grids; "heavy_prio" (default 1): heavy tier on a
 * highest-priority stream; "warp" (default 1): bulk tier with one WARP per problem (k_warp.cu; 0 = one CTA per problem);
 * "warp_cfg" (default 3): its CTA shape (0: 12 warps x 1 CTA/SM, 1: 3 x 3, 2: 4 x 3, 3: 1 x 10, 4: 2 x 5); "warp_zs"
 * (default 0 = as many as fit): cached directions per warp kept in shared memory; "screen" (default 2, 0..3): number of screening
 * passes -- outer iterations 1..screen of the warp tier run in launches of their own, each followed by a heavy-tier launch for
 * the long dual chains it found (on the high-priority stream, concurrent with the rest of the work); "heavy_cfg" (default 0):
 * 1 = slim heavy tier (64 x 64 inverse on chip, 168 registers); "warp_qcap" (default 15): rows a working set may reach in
 * the warp tier before the problem goes to the heavy tier; "one_shot", "warp_lockstep", "heavy_skip": measurement switches
 * (DESIGN.md section 4b). */
int cfs_set_option(cfs_ctx *ctx, const char *name, int value);

/* ---- problem data ------------------------------------------------------------------------------------- */
/* robotproperty2.m:12-139 -> sys_info.robot.{DH (6x4), base (3), cap{i}.p (3x2 per link), delta_t}; T2L = robot.T
 * (3x3, only for CFS_ROBOT_2L, else NULL).  n_joints = sys_info.njoint (links used = first n_joints rows). */
int cfs_set_robot(cfs_ctx *ctx, int robot_kind, const double *DH /*6x4*/, int dh_rows, const double *base /*3*/,
                  const double *cap_p /*3x2xn_joints*/, int n_joints, const double *T2L /*3x3 or NULL*/, double dt);
/* obs{j}.l (3x2), obs{j}.D, obs{j}.epsilon   (main_FANUC.m:56-60) */
int cfs_set_obstacles(cfs_ctx *ctx, const double *seg /*3x2xn_obs*/, const double *D, const double *eps, int n_obs);
/* The same with a kind per obstacle (NULL = all capsules).  CFS_OBS_CAPSULE: seg(:,:,j) = obs{j}.l, the capsule axis -- the
 * only obstacle the reference has.  CFS_OBS_BOX (extension, SURVEY.md section 8f N3; MATLAB side: obs{j}.shape = 'box'):
 * seg(:,1,j) / seg(:,2,j) = min / max corner of a solid axis-aligned box, e.g. the bounding box of an STL part of map/
 * (Lib/functions/MapFromSTL.m:1-12 reads those, in mm).  The distance is taken between the link AXIS and the solid box, with
 * the same "|dis| < 1e-4 -> -norm(P1 - link end)" rule and the same margins D / epsilon as for capsules. */
enum { CFS_OBS_CAPSULE = 0, CFS_OBS_BOX = 1 };
int cfs_set_obstacles_ex(cfs_ctx *ctx, const double *seg /*3x2xn_obs*/, const int *kind /*n_obs or NULL*/, const double *D,
                         const double *eps, int n_obs);
/* sys_info.{H, QQ, lim, MAX_input} (main_FANUC.m:106-127).  lim==NULL: no velocity rows (M16iB/main_CFS.m path);
 * max_input==NULL: no bounds.  Factors QQ once on the device and builds the shared Gram operator. */
int cfs_set_cost(cfs_ctx *ctx, int H, const double *QQ /*n x n, n=H*n_joints*/, const double *lim /*n_joints*/,
                 const double *max_input /*n*/);

/* Joint position limits (extension: the reference has none, robotproperty2.m).  qmin / qmax: n_joints entries each, or both
 * NULL to clear the limits.  qmin_k may be -INFINITY and qmax_k +INFINITY for a joint without that side.  CFS_E_ARG if only
 * one pointer is NULL, an entry is NaN, qmin_k > qmax_k, qmin_k = +INFINITY or qmax_k = -INFINITY (a limit no position meets);
 * CFS_E_STATE without a robot.  cfs_set_robot clears the limits.
 * With limits set, the QP of every CFS and PSGCFS solve (cfs_solve_batch*, cfs_solve_start_goal*, cfs_solve_routes*,
 * cfs_solve_batch_margins*, every round of cfs_solve_checked*; both gradient modes) also has, for every waypoint i = 1..H and
 * joint k, the rows theta_i,k <= qmax_k and -theta_i,k <= -qmin_k, theta_i the roll-out of u from x0 (waypoint 0 is x0 and is
 * not constrained); an infinite bound gives a row that can never be violated.  Nothing else changes: stop rule, cost, status
 * codes, the reference's rows.  The limits hold at the waypoints only: theta is quadratic on a segment and may overshoot a
 * limit both of its ends satisfy.  A start outside the limits gives what the QP gives, normally CFS_STATUS_INFEASIBLE.
 * cfs_get_con appends the 2n rows (upper rows, then lower rows, [waypoint][joint] order).  cfs_chomp_batch, the unconstrained
 * baseline, does not read the limits. */
int cfs_set_joint_limits(cfs_ctx *ctx, const double *qmin /*n_joints or NULL*/, const double *qmax /*n_joints or NULL*/);

/* Same as cfs_set_cost with QQ built ON THE DEVICE from the blocks the mains assemble it from (main_FANUC.m:64-97,
 * RRTstar_CFS.m:124-160, main_2L.m:69-92): QQ = Baug'*Qaug*Baug + r_scale*(R+R'), Qaug = blkdiag(stage_w*Q ... term_w*Q),
 * R = blkdiag(Rblk).  Enables cfs_solve_start_goal.  (SURVEY.md section 8f, N2.) */
int cfs_set_cost_blocks(cfs_ctx *ctx, int H, const double *Q /*2nj x 2nj*/, const double *Rblk /*nj x nj*/, double r_scale,
                        double stage_w, double term_w, const double *lim /*nj or NULL*/, const double *max_input /*n or NULL*/);

/* ---- the hot path ------------------------------------------------------------------------------------- */
/* CFS_FANUC.optimizer (Lib/CFS_FANUC.m:62-79) / PSGCFS_FANUC.optimizer (Lib/PSGCFS_FANUC.m:65-82) for B problems.
 *   x0 = sys_info.xR(:,1), ff = sys_info.ff, caug = sys_info.caug, xref = sys_info.x_, noise = the normrnd draws of
 *   PSGCFS_FANUC.m:109 (n x max_outer x B, iteration-major per problem; NULL = zeros), alpha = sys_info.alpha.
 *   outputs: u = self.u, x = self.x_, cost_hist = self.eval.cost_all (NaN padded), e_u_hist = self.eval.e_u_all,
 *   iters = self.iter_O-1, status as above.  e_u_hist may be NULL. */
int cfs_solve_batch(cfs_ctx *ctx, int B, int solver, int grad, const double *x0 /*2nj x B*/, const double *ff /*n x B*/,
                    const double *caug /*B*/, const double *xref /*2njH x B*/, const double *noise, double eps_outer,
                    int max_outer, double alpha, double *u /*n x B*/, double *x /*2njH x B*/,
                    double *cost_hist /*max_outer x B*/, double *e_u_hist /*max_outer x B or NULL*/, int *iters /*B*/,
                    int *status /*B*/);
/* Asynchronous form of cfs_solve_batch: enqueues H2D copies, the solve and the D2H copies on the context stream and
 * returns.  The host buffers must stay valid (and should be pinned for the copies to overlap other contexts' kernels)
 * until cfs_wait(ctx) returns.  One batch may be in flight per context; several contexts on one device pipeline
 * copy(k+1) | solve(k) | copy(k-1)  -- the GPU analogue of the reference's parfor workers (s_Parallel_rrt.m:16). */
int cfs_solve_batch_async(cfs_ctx *ctx, int B, int solver, int grad, const double *x0, const double *ff, const double *caug,
                          const double *xref, const double *noise, double eps_outer, int max_outer, double alpha, double *u,
                          double *x, double *cost_hist, double *e_u_hist, int *iters, int *status);
/* The mains' problem set-up + optimizer() for B start/goal pairs (main_FANUC.m:38-49: x0 = [theta0; 0], x_ = straight line
 * in joint space, zero velocity rows; :98-103: gaug = [thetag; 0] tiled, ff, caug), built on the device: 80 B in per problem
 * instead of 6 KB.  Needs cfs_set_cost_blocks.  x and e_u_hist may be NULL (then not copied back). */
int cfs_solve_start_goal(cfs_ctx *ctx, int B, int solver, int grad, const double *theta0 /*nj x B*/, const double *thetag /*nj x B*/,
                         const double *noise, double eps_outer, int max_outer, double alpha, double *u, double *x,
                         double *cost_hist, double *e_u_hist, int *iters, int *status);
int cfs_solve_start_goal_async(cfs_ctx *ctx, int B, int solver, int grad, const double *theta0, const double *thetag,
                               const double *noise, double eps_outer, int max_outer, double alpha, double *u, double *x,
                               double *cost_hist, double *e_u_hist, int *iters, int *status);
/* RRT*-CFS glue (RRTstar_CFS.m:96-119, SURVEY.md section 8f N1), on the device: every route (nj x W waypoints, dt apart) is
 * resampled to H+1 points with cubicpolytraj's default boundary conditions (zero velocity at every waypoint:
 * q = q_k + (3s^2 - 2s^3)(q_{k+1} - q_k) on segment k), x0 = [sample_1; 0], xg = sample_{H+1}, x_ = [sample_i; 0] (i = 2..H+1),
 * ff / caug as in cfs_solve_start_goal, then optimizer().  Needs cfs_set_cost_blocks.  (cubicpolytraj is Robotics System
 * Toolbox code, not part of the reference tree: parity unpinned, see DESIGN.md.) */
int cfs_solve_routes(cfs_ctx *ctx, int B, int W, int solver, int grad, const double *routes /*nj x W x B*/, const double *noise,
                     double eps_outer, int max_outer, double alpha, double *u, double *x, double *cost_hist, double *e_u_hist,
                     int *iters, int *status);
int cfs_solve_routes_async(cfs_ctx *ctx, int B, int W, int solver, int grad, const double *routes, const double *noise,
                           double eps_outer, int max_outer, double alpha, double *u, double *x, double *cost_hist,
                           double *e_u_hist, int *iters, int *status);
/* The same for routes of different lengths (one per RRT seed: Lib/functions/s_Parallel_rrt.m:16-25): routes is nj x W x B with
 * the first route_len[b] columns of problem b valid.  route_len[b] < 2 (failed seed): status CFS_STATUS_NO_ROUTE. */
int cfs_solve_routes_var(cfs_ctx *ctx, int B, int W, const int *route_len /*B*/, int solver, int grad, const double *routes,
                         const double *noise, double eps_outer, int max_outer, double alpha, double *u, double *x,
                         double *cost_hist, double *e_u_hist, int *iters, int *status);
int cfs_solve_routes_var_async(cfs_ctx *ctx, int B, int W, const int *route_len, int solver, int grad, const double *routes,
                               const double *noise, double eps_outer, int max_outer, double alpha, double *u, double *x,
                               double *cost_hist, double *e_u_hist, int *iters, int *status);
/* ... every pointer a DEVICE pointer (route_len may be NULL: all routes have W waypoints); asynchronous unless sync != 0.
 * Chains with cfs_rrt_find_routes_device without a host round trip: the RRT -> CFS pipeline of RRTstar_CFS.m:76-195. */
int cfs_solve_routes_device(cfs_ctx *ctx, int B, int W, const int *route_len, int solver, int grad, const double *routes,
                            const double *noise, double eps_outer, int max_outer, double alpha, double *u, double *x,
                            double *cost_hist, double *e_u_hist, int *iters, int *status, int sync);
/* The resampling step alone: sampled (nj x (H+1) x B) = cubicpolytraj(route, (0:W-1)*dt, linspace(0,(W-1)*dt,H+1)). */
int cfs_resample_routes(cfs_ctx *ctx, int B, int W, int H, const double *routes /*nj x W x B*/, double *sampled);
/* CHOMP_FANUC(obs, sys_info, uu, ROBOT).optimizer()  (Lib/CHOMP_FANUC.m:54-165), the gradient-descent baseline planner of the
 * reference (SURVEY.md section 8f, N4), for B problems that share robot, obstacles and cost.  Unconstrained: it does not
 * read the joint limits of cfs_set_joint_limits.
 *   u_init = uu (n x B), xref = sys_info.x_, alpha = sys_info.alpha; obs{j}.D / obs{j}.epsilon from cfs_set_obstacles.
 *   Every outer iteration: dm_f per link (:115-134), derivest gradient of dist_link_*(linkid) (:151,:156), the update
 *   u <- u - alpha*3*(QQ*u + ff + 2000*dcostObs) (:75), roll-out, cost_all(k) = get_cost(u) + fobs_m() (:63).
 *   The reference's stop rule never fires before MAX_O_ITER (eval.x_ / eval.x_old are never updated by this class), so
 *   iters = max_outer and status = CFS_STATUS_MAX_ITER for every problem (| CFS_FLAG_TOUCH).  x and e_u_hist may be NULL.
 *   Two quirks of the reference are reproduced as written and documented in DESIGN.md: dm_f has no joint-2 offset on the
 *   200i, and the gradient of waypoint i is chained through Baug((i-1)*njoint+1 : i*njoint, :) (row stride njoint). */
int cfs_chomp_batch(cfs_ctx *ctx, int B, const double *x0 /*2nj x B*/, const double *ff /*n x B*/, const double *caug /*B*/,
                    const double *xref /*2njH x B*/, const double *u_init /*n x B*/, double alpha, int max_outer,
                    double *u /*n x B*/, double *x /*2njH x B or NULL*/, double *cost_hist /*max_outer x B*/,
                    double *e_u_hist /*max_outer x B or NULL*/, int *iters /*B*/, int *status /*B*/);

/* Blocks until the context's stream is idle and collects the statistics of the batch in flight (if any). */
int cfs_wait(cfs_ctx *ctx);
/* Same, every pointer is a DEVICE pointer on ctx's device (inputs already resident in HBM); asynchronous on the
 * context stream unless sync != 0. */
int cfs_solve_batch_device(cfs_ctx *ctx, int B, int solver, int grad, const double *x0, const double *ff,
                           const double *caug, const double *xref, const double *noise, double eps_outer,
                           int max_outer, double alpha, double *u, double *x, double *cost_hist, double *e_u_hist,
                           int *iters, int *status, int sync);

/* dist_arm_all + gradient for N configurations against every obstacle
 * (CFS_FANUC.m:115-118: dist_arm_3D_Heu_2 / dist_arm_3D_200i_2 / dist_arm_2L + num_jac, or derivest+dist_link_*).
 *   dist (n_obs x N), linkid (n_obs x N, 1-based), grad (nj x n_obs x N), flags (N: CFS_FLAG_TOUCH or 0). */
int cfs_dist_grad(cfs_ctx *ctx, int N, int grad_mode, const double *theta /*nj x N*/, double *dist, int *linkid,
                  double *grad, int *flags);

/* Times the stand-alone distance/gradient kernel (K1 / K1d) on N configurations resident in HBM: theta is uploaded once
 * (untimed), 2 warm-up launches, then `reps` launches bracketed by CUDA events on the context stream. */
int cfs_time_dist_grad(cfs_ctx *ctx, int N, int grad_mode, const double *theta /*nj x N*/, int reps, double *ms_per_launch);

/* CFS_FANUC.get_con (Lib/CFS_FANUC.m:101-135) for ONE problem, dense and in the reference's row order
 * (per obstacle j, step i: 1 obstacle row, nj rows +Baug_w, nj rows -Baug_w).  Ainq is m x n column-major,
 * m = n_obs*H*(1+2nj) (or n_obs*H when no lim was set), plus 2n joint position rows after them when joint limits are set
 * (cfs_set_joint_limits).  margin_is_D: 0 -> obs.epsilon (CFS), 1 -> obs.D (PSGCFS). */
int cfs_get_con(cfs_ctx *ctx, int grad_mode, int margin_is_D, const double *x0, const double *xcur /*2njH*/,
                const double *u /*n*/, double *Ainq, double *binq);

/* RRT_FANUC.feasible (Lib/RRT_FANUC.m:146-181) for N candidate nodes: feasible[i]=1 iff every link distance to every
 * obstacle is >= obs.D; dmin = min distance over links and obstacles. */
int cfs_nodes_feasible(cfs_ctx *ctx, int N, const double *theta /*nj x N*/, unsigned char *feasible, double *dmin);
/* ---- continuous collision checks (extension: the reference checks RRT nodes only, RRT_FANUC.m:129,146-181) ------------
 * Clearance of a configuration: c(theta) = min over links l and obstacles j of (d_lj(theta) - m_j), d_lj the link-axis distance
 * of cfs_nodes_feasible / cfs_dist_grad (capsules and boxes, "axes touch" rule included), m_j = obs{j}.D if margin_is_D != 0,
 * else obs{j}.epsilon.  At one configuration the hit test gives exactly the verdict of cfs_nodes_feasible.
 * Paths: an edge is theta(s) = theta_a + s (theta_b - theta_a), s in [0, 1] (RRT edges, route polylines); segment k of a
 * trajectory is the double integrator between its waypoints, theta(tau) = theta_k + omega_k tau + (tau^2 / 2) u_k, tau in
 * [0, dt], from state x_k (x0 for k = 0) with control u_k -- exact for CFS trajectories (A = [I dt I; 0 I], B = [dt^2/2 I; dt I]).
 * Motion bound: cfs_set_robot computes per joint R_j >= ||dp/dtheta_j|| for every link-axis endpoint p of the links l >= j at
 * every theta (triangle inequality over the DH / robot.T translations and the capsule endpoints), so that
 * |c(theta1) - c(theta2)| <= sum_j R_j TV_j (TV_j: total variation of joint j between them).
 * Algorithm (conservative advancement, tolerance eta > 0), sequential per item:
 *   vmax = sum_j R_j |theta_b,j - theta_a,j| (edge), sum_j R_j max(|omega_j|, |omega_j + u_j dt|) (segment);
 *   s = 0; loop: evaluate c(s); c < -eta/2 -> HIT at s; s at the end (or vmax == 0) -> CLEAR;
 *   else s += (c + eta) / vmax, clamped to the end.  More than max_evals evaluations needed -> UNDECIDED.
 * Guarantees: a CLEAR item has c >= -eta along its whole path; a HIT item has a witness with c < -eta/2 and c >= -eta before it.
 * So an item whose true minimum is >= -eta/2 is CLEAR, one below -eta is HIT; the eta/2 threshold keeps waypoints that the
 * linearised CFS constraint leaves ~1e-9 below the margin from counting as hits.  CFS_E_ARG unless eta > 0 and
 * min_j m_j - eta >= 1e-4 (the touch rule then never fires inside the certified band) and max_evals >= 1.  No robot or
 * obstacles yet: CFS_E_STATE.  N = 0 / B = 0: no-op.  Results are deterministic (no order-dependent reduction). */
enum { CFS_CHECK_CLEAR = 0, CFS_CHECK_HIT = 1, CFS_CHECK_UNDECIDED = 2 };
/* per edge: verdict, s_hit (-1 if none), cmin = smallest c evaluated, evals (may be NULL) */
int cfs_check_edges(cfs_ctx *ctx, int N, const double *theta_a /*nj x N*/, const double *theta_b /*nj x N*/, double eta,
                    int margin_is_D, int max_evals, int *verdict, double *s_hit, double *cmin, int *evals);
/* per trajectory (x must be the roll-out of u, as every solve entry returns it): verdict = HIT if any segment hits, else
 * UNDECIDED if any segment is, else CLEAR; t_hit = earliest hit time in [0, H dt] (k dt + tau, -1 if none); cmin = min over
 * segments; evals = sum over segments (may be NULL) */
int cfs_check_trajectories(cfs_ctx *ctx, int B, int H, const double *x0 /*2nj x B*/, const double *x /*2njH x B*/,
                           const double *u /*njH x B*/, double eta, int margin_is_D, int max_evals, int *verdict,
                           double *t_hit, double *cmin, int *evals);
/* the same with every pointer a DEVICE pointer; asynchronous on the context stream unless sync != 0 */
int cfs_check_edges_device(cfs_ctx *ctx, int N, const double *theta_a, const double *theta_b, double eta, int margin_is_D,
                           int max_evals, int *verdict, double *s_hit, double *cmin, int *evals, int sync);
int cfs_check_trajectories_device(cfs_ctx *ctx, int B, int H, const double *x0, const double *x, const double *u, double eta,
                                  int margin_is_D, int max_evals, int *verdict, double *t_hit, double *cmin, int *evals,
                                  int sync);

/* ---- per-waypoint margin offsets and the checked solve ----
 * cfs_solve_batch_margins: cfs_solve_batch plus margin_off (nobs x H per problem: element (b nobs + j) H + (i - 1) for
 * waypoint i = 1..H, the [prob][obs][i] order; NULL = no offsets).  The obstacle row of (obstacle j, waypoint i) becomes
 * dist - (m_j + margin_off) instead of dist - m_j (m_j = epsilon for CFS, D for PSGCFS); nothing else changes, and all-zero
 * offsets give bit for bit the result of cfs_solve_batch.  Entries must be finite and >= 0 (CFS_E_ARG).  The _device form checks
 * them on the device and synchronises once for that.  Uses: time-varying clearance, and the repair of cfs_solve_checked.
 *
 * cfs_solve_checked: a solve whose trajectories come back with a continuous collision check, after repairing the ones that
 * cut an obstacle margin between waypoints (CFS constrains the waypoints only).  The check margin is the solver's (epsilon for
 * CFS, D for PSGCFS); eta, max_evals as in cfs_check_trajectories (same argument rules); rounds >= 0; gain > 0 and finite.
 *   Round 0 is exactly cfs_solve_batch_device followed by cfs_check_trajectories_device.
 *   After each check, every problem whose current verdict is HIT and whose status low byte is < 2 gets, for each HIT segment k
 *   with witness theta* (the point where the check found c < -eta/2) and each obstacle j with clearance c_j(theta*) < -eta/2,
 *   inc = gain (eta - c_j) at waypoints k and k+1 (those in 1..H; waypoint 0 is x0); a waypoint between two HIT segments gets
 *   the larger increment, not the sum.  The increments add to its offsets (starting at 0).
 *   Round r = 1..rounds re-solves those problems from the caller's original xref with their accumulated offsets.  A candidate
 *   whose status low byte is < 2 replaces the problem's solution and is checked again; a failed one (INFEASIBLE / NUMERICAL)
 *   leaves the previous solution, and the problem stops repairing.  Problems with status >= 2 after round 0 are returned as
 *   round 0 left them.  The loop ends after `rounds` rounds or when no problem is left to repair.
 * Outputs: u, x, cost_hist, e_u_hist (may be NULL), iters, status of the returned solution; verdict, t_hit, cmin of its check;
 * rounds_used = the round that produced it (0 = the first solve); margin_off (may be NULL): the offsets that returned solution
 * was solved with (0 where rounds_used is 0), so cfs_solve_batch_margins with them reproduces it.  A CLEAR verdict carries the
 * guarantee of cfs_check_trajectories.
 * Each round reads one count back from the device, and the statistics of round 0 are collected, so the _device form
 * synchronises after round 0 and once per round.  cfs_get_stats describes round 0's solve.  The host form is synchronous. */
int cfs_solve_batch_margins(cfs_ctx *ctx, int B, int solver, int grad, const double *x0, const double *ff, const double *caug,
                            const double *xref, const double *noise, const double *margin_off /*nobs H x B or NULL*/,
                            double eps_outer, int max_outer, double alpha, double *u, double *x, double *cost_hist,
                            double *e_u_hist, int *iters, int *status);
int cfs_solve_batch_margins_device(cfs_ctx *ctx, int B, int solver, int grad, const double *x0, const double *ff,
                                   const double *caug, const double *xref, const double *noise, const double *margin_off,
                                   double eps_outer, int max_outer, double alpha, double *u, double *x, double *cost_hist,
                                   double *e_u_hist, int *iters, int *status, int sync);
int cfs_solve_checked(cfs_ctx *ctx, int B, int solver, int grad, const double *x0, const double *ff, const double *caug,
                      const double *xref, const double *noise, double eps_outer, int max_outer, double alpha, double eta,
                      int max_evals, int rounds, double gain, double *u, double *x, double *cost_hist, double *e_u_hist,
                      int *iters, int *status, int *verdict /*B*/, double *t_hit /*B*/, double *cmin /*B*/,
                      int *rounds_used /*B*/, double *margin_off /*nobs H x B or NULL*/);
int cfs_solve_checked_device(cfs_ctx *ctx, int B, int solver, int grad, const double *x0, const double *ff, const double *caug,
                             const double *xref, const double *noise, double eps_outer, int max_outer, double alpha, double eta,
                             int max_evals, int rounds, double gain, double *u, double *x, double *cost_hist, double *e_u_hist,
                             int *iters, int *status, int *verdict, double *t_hit, double *cmin, int *rounds_used,
                             double *margin_off, int sync);
/* RRT_FANUC.getRandNode nearest scan + steer (Lib/RRT_FANUC.m:116-129) for S samples against one tree:
 * parent[s] = argmin_i ||(nodes(:,i)-sample(:,s)).*ratial|| (first minimum, 0-based), newnode = parent + (sample-parent)*step/||parent-sample||. */
int cfs_nearest_steer(cfs_ctx *ctx, int n_nodes, const double *nodes /*nj x n_nodes*/, int S, const double *samples /*nj x S*/,
                      const double *ratial /*nj*/, double step, int *parent /*S*/, double *newnode /*nj x S*/);
/* RRT_FANUC.find_route (Lib/RRT_FANUC.m:63-207: getNode / getRandNode / feasible / addNode / arrangeNode / goal_reached) for
 * S independent seeds at once -- the parfor over num_seed workers of Lib/functions/s_Parallel_rrt.m:16-25 -- one CTA per seed,
 * trees in shared memory (SURVEY.md section 8f, N4).  star != 0: 'RRT*' (re-parenting), else 'RRT'.  MATLAB's rand stream is an
 * input: rnd (nrnd x S) is consumed per seed in the reference's order (pp = rand; rand(nstate,1) when pp < bi).
 *   x0 / goal / goal_th: nj x S (sys_info.x0, goalxyz, sys_info.goal_th); region_g, region_s, sample_off, ratial: nj; bi = 0.5,
 *   max_iter = 400 in the reference (RRT_FANUC.m:37-38).  Obstacles and their D come from cfs_set_obstacles.
 *   routes: nj x (max_iter+2) x S, the first route_len[s] columns are self.route; route_len = size(route,2) = routeL
 *   (-1: rnd exhausted); n_nodes = node_num; fail = self.fail; rnd_used = numbers consumed.  tree_* (nj x (max_iter+2) x S,
 *   (max_iter+2) x S; all three or none) receive all_nodes(2:end,:), all_nodes(1,:) and total_dis; ms_kernel may be NULL. */
int cfs_rrt_find_routes(cfs_ctx *ctx, int S, int star, const double *x0, const double *goal, const double *goal_th,
                        const double *region_g, const double *region_s, const double *sample_off, const double *ratial,
                        double bi, int max_iter, const double *rnd, int nrnd, double *routes, int *route_len, int *n_nodes,
                        int *fail, int *rnd_used, double *tree_nodes, int *tree_parent, double *tree_total, double *ms_kernel);

/* cfs_rrt_find_routes with every array in device memory (params = [region_g; region_s; sample_off; ratial], 4*nj doubles);
 * asynchronous on the context stream unless sync != 0.  A failed seed reports route_len as found by the back-trace and
 * fail = 1; use route_len_or_fail (S ints, may be NULL) to get 0 for failed / exhausted seeds, ready for
 * cfs_solve_routes_device. */
int cfs_rrt_find_routes_device(cfs_ctx *ctx, int S, int star, const double *x0, const double *goal, const double *goal_th,
                               const double *params, double bi, int max_iter, const double *rnd, int nrnd, double *routes,
                               int *route_len, int *n_nodes, int *fail, int *rnd_used, int *route_len_or_fail, int sync);

/* ---- introspection (profiling / bench) ---------------------------------------------------------------- */
typedef struct {
  double ms_setup;        /* last cfs_set_cost: device factorisation time                                 */
  double ms_total;        /* last cfs_solve_batch*: device time of the whole solve (CUDA events)          */
  double ms_grad;         /* ... of the distance/gradient kernel launches                                 */
  double ms_qp;           /* ... of the QP/rollout kernel launches                                        */
  double ms_h2d, ms_d2h;  /* ... of its H2D / D2H copies when a host-pointer form ran it, 0 for a _device form */
  long long grad_waypoints; /* (problem, waypoint, obstacle) gradient evaluations done                    */
  long long problem_iters;  /* sum over problems of outer iterations                                      */
  long long qp_steps;       /* sum of dual active-set iterations                                          */
  int launches;           /* kernels launched by the last solve                                           */
  int max_active;         /* largest working set seen                                                     */
  double ms_bulk, ms_heavy; /* timing level 2, fused kernel: device time of its bulk / heavy tier launch        */
} cfs_stats;
int cfs_get_stats(const cfs_ctx *ctx, cfs_stats *out);
/* level 1 (default): whole-solve time only; level 2: per-kernel CUDA events (ms_grad / ms_qp) */
int cfs_set_timing(cfs_ctx *ctx, int level);
/* per-outer-iteration kernel times of the last level-2 solve: grad_ms[k], qp_ms[k], k < min(cap, max_outer); returns count */
int cfs_get_iter_times(const cfs_ctx *ctx, double *grad_ms, double *qp_ms, int cap);
/* dual active-set steps spent on each problem of the last solve (sum over outer iterations), steps[B] */
int cfs_get_problem_steps(cfs_ctx *ctx, int *steps, int B);
/* timing level 3: clock64 phase profile of the QP kernel (thread 0 of every CTA, summed): out8 = {prologue, primal
 * refresh, violation scan, gram+solve+step length, working-set update, epilogue} ticks, problems, outer steps; out16[8..15]
 * = the same for the heavy tier of the fused kernel */
int cfs_get_qp_profile(cfs_ctx *ctx, long long *out16);
/* timing level 3, warp tier (nj = 5, one obstacle, default CTA shape): clock64 cycles summed over the warps of the last solve:
 * out6 = {gradient phase (get_con: FK + distances + num_jac), QP (mask + dual active set), whole problems, gradient passes,
 *         warps resident on the device with a full grid, SMs}.
 * The gradient code's own rate -- what the kernel would sustain if every resident warp were in its gradient phase -- is
 *   passes * H * n_obs * 9680 FLOP / (out6[0] / out6[4]) cycles; bench.py reports it as roofline.gradient_phase. */
int cfs_get_warp_profile(cfs_ctx *ctx, long long *out6);
/* FP64 FMA micro-benchmark (roofline denominator: MEASURED_PEAKS.json has no FP64 entry). Returns TFLOP/s. */
int cfs_measure_fp64_peak(cfs_ctx *ctx, double *tflops, double *sm_clock_mhz_est);

#ifdef __cplusplus
}
#endif
#endif
