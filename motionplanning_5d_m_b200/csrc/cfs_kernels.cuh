// cfs_kernels.cuh -- launch wrappers shared between the translation units of libcfs_b200.
#pragma once
#include <cuda_runtime.h>

#include "cfs_types.cuh"

namespace cfs {

// ---- K1 / K1d : distance + gradient ---------------------------------------------------------------------
// Work item = (slot, i): configuration theta = x[prob*ld_prob + i*ld_i + k], k < nj, prob = list ? list[slot] : slot.
// Outputs for obstacle j:   dist[prob*o_prob + j*o_obs + i*o_i], linkid (same index), grad[(same index)*nj + k].
struct GradArgs {
  const DevTables *tab;
  const DerivestTab *dv;     // K1d only
  const double *x;
  long long ld_prob, ld_i;
  const int *list;           // active problem list or nullptr
  const int *count;          // device-side number of active slots or nullptr (=> nslots)
  int nslots;                // upper bound on slots
  int H;                     // configurations per problem
  int nj, nobs;
  long long o_prob, o_obs, o_i;
  double *dist;
  int *linkid;
  double *grad;
  int *flags;                // per problem: OR of CFS_FLAG_TOUCH (atomicOr)
  // K1d, CHOMP_FANUC.dm_f mode (Lib/CHOMP_FANUC.m:115-134): the base evaluation (distance per link, linkid) ignores the joint
  // offsets of the table (dm_f sets DH(i,1) = theta(i) and nothing else, also on the 200i), the derivest evaluations of
  // dist_link_* keep them; linkdist (or nullptr) receives the nj per-link distances of every (waypoint, obstacle) pair
  int no_off;
  double *linkdist;
};
cudaError_t launch_grad_numjac(const GradArgs &a, cudaStream_t s);
cudaError_t launch_grad_derivest(const GradArgs &a, cudaStream_t s);

// ---- K6 : RRT node feasibility and nearest/steer ----------------------------------------------------------
cudaError_t launch_nodes_feasible(const DevTables *tab, int nj, int nobs, int N, const double *theta,
                                  unsigned char *feasible, double *dmin, cudaStream_t s);
cudaError_t launch_nearest_steer(int nj, int n_nodes, const double *nodes, int S, const double *samples,
                                 const double *ratial, double step, int *parent, double *newnode, cudaStream_t s);

// ---- continuous collision checks of edges / trajectory segments (k_check.cu) ------------------------------------------------
enum { CHK_CLEAR = 0, CHK_HIT = 1, CHK_UNDECIDED = 2 };  // = CFS_CHECK_* of include/cfs_b200.h
struct CheckArgs {
  const DevTables *tab;
  int mode;                        // 0: edges, 1: trajectory segments (item = b*H + k)
  int N, H, nj, nobs, margin_is_D, max_evals;
  double eta;
  double R[CFS_MAXL];              // motion bound per joint (cfs_set_robot); a kernel argument, not part of DevTables
  const double *theta_a, *theta_b; // mode 0: nj x N
  const double *x0, *x, *u;        // mode 1: 2nj x B, 2njH x B, njH x B
  int *verdict;                    // per item
  double *s_hit, *cmin;
  int *evals;                      // per item, may be nullptr
  int *counter;                    // work queue head (zeroed by launch_check)
};
cudaError_t launch_check(const CheckArgs &a, int device, cudaStream_t s);
// per-segment results (B*H each) -> per-trajectory verdict, t_hit, cmin, evals (evals may be nullptr)
cudaError_t launch_check_reduce(int B, int H, double dt, const int *sv, const double *ss, const double *sc, const int *se,
                                int *verdict, double *t_hit, double *cmin, int *evals, cudaStream_t s);
// repair increments of the checked solve: per trajectory b, segments in order; for every HIT segment k the witness theta* of
// s_hit[k] and its clearance per obstacle c_j; obstacles with c_j < -eta/2 get inc = gain (eta - c_j) at waypoints k and k+1
// (1..H only), the maximum over the adjacent HIT segments, added to margin_off[(b nobs + j) H + i - 1].  a.verdict / a.s_hit
// are the per-segment results of launch_check (mode 1); x0 / x / u the checked trajectories.
// sel[t] (t < *count, at most nmax) are positions in the checked set, map[pos] (nullptr: identity) the problem of margin_off
cudaError_t launch_repair_margins(const CheckArgs &a, int nmax, const int *count, const int *sel, const int *map, double gain,
                                  double *margin_off, cudaStream_t s);
// the round loop of the checked solve: stable selection of the positions p < N with verdict[p] == HIT and status low byte < 2
// (sel = positions, next = map[p] or p, *count); row gather (dst[t] = src[list[t]]) / scatter (dst[list[t]] = src[t], skipped
// where st[t] low byte >= 2); fill >= 0 writes that value instead of src
cudaError_t launch_repair_select(int N, const int *verdict, const int *status, const int *map, int *sel, int *next, int *count,
                                 cudaStream_t s);
cudaError_t launch_rows_copy(int n_rows, const int *list, const double *src, double *dst, long long len, int scatter, const int *st,
                             cudaStream_t s);
cudaError_t launch_ints_copy(int n_rows, const int *list, const int *src, int *dst, int scatter, const int *st, int fill,
                             cudaStream_t s);
cudaError_t launch_offsets_bad(long long N, const double *off, int *bad, cudaStream_t s);

// work order of the fused solver (longest expected problems first): order[] = problems by descending number of reference
// waypoints inside an obstacle margin; count[] is scratch (B ints each)
cudaError_t launch_work_order(const DevTables *tab, int nj, int nobs, int B, int H, const double *xref, int margin_is_D,
                              int *count, int *order, cudaStream_t s);

// ---- batched RRT / RRT* tree growth, one CTA per seed (k_rrt.cu) -------------------------------------------------------------
struct RrtArgs {
  const DevTables *tab;
  int nj, nobs, star, max_iter, nrnd;
  double bi;
  const double *x0, *goal, *goal_th;                          // nj x S
  const double *region_g, *region_s, *sample_off, *ratial;    // nj
  const double *rnd;                                          // nrnd x S uniform numbers, consumed in MATLAB's order
  double *routes;                                             // nj x (max_iter+2) x S
  int *route_len, *n_nodes, *fail, *rnd_used;                 // S   (route_len = -1: random stream exhausted)
  double *tree_nodes, *tree_total;                            // optional: nj x (max_iter+2) x S, (max_iter+2) x S
  int *tree_parent;                                           // optional: (max_iter+2) x S
};
cudaError_t launch_rrt_find_routes(const RrtArgs &a, int S, cudaStream_t s);

// ---- set-up: shared Gram operator G = P QQ^{-1} P' ----------------------------------------------------------
// P = [B_theta; B_omega; I] (3n x n): the primitives every constraint row of CFS_FANUC.get_con is built from.
// hessian_is_identity: PSGCFS projection (PSGCFS_FANUC.m:117) -> G = P P'.
cudaError_t setup_gram(int n, int H, int nj, double dt, const double *QQ /*device n x n or nullptr*/, double *work_L /*n*n*/,
                       double *work_Y /*n*3n*/, double *G /*3n x 3n*/, double *gdiag /*3n*/, int *info /*device*/,
                       cudaStream_t s);

// ---- problem set-up on the device (SURVEY.md section 8f, N2) ------------------------------------------------------------
// QQ = Baug'*Qaug*Baug + r_scale*(R+R') of main_FANUC.m:64-97 from its blocks: Q (2nj x 2nj stage cost, weight stage_w on
// steps 1..H-1 and term_w on step H), Rblk (nj x nj).  Baug's blocks are closed form ((0.5+(i-j))dt^2 I ; dt I).
cudaError_t launch_build_qq(int H, int nj, double dt, const double *Q, const double *Rblk, double r_scale, double stage_w,
                            double term_w, double *QQ /*n x n*/, cudaStream_t s);
// per problem, from a start/goal pair (main_FANUC.m:38-49, 98-103): x0 = [theta0; 0], x_ = straight line in joint space
// with zero velocity rows (step 0 dropped), gaug = [thetag; 0] tiled, ff = ((Aaug x0 - gaug)' Qaug Baug)', caug = e' Qaug e
cudaError_t launch_build_problems(int B, int H, int nj, double dt, const double *Q, double stage_w, double term_w,
                                  const double *theta0 /*nj x B*/, const double *thetag /*nj x B*/, double *x0 /*2nj x B*/,
                                  double *xref /*2njH x B*/, double *ff /*n x B*/, double *caug /*B*/, cudaStream_t s);

// RRT route (nj x W waypoints dt apart) -> H+1 samples of cubicpolytraj with zero waypoint velocities (RRTstar_CFS.m:96-100):
// theta0 / thetag = first / last sample, xref = [sample_i; 0], i = 1..H.  launch_build_problems with xref == nullptr then
// adds x0, ff, caug without touching that reference.
// route_len (B, or nullptr: every route has W waypoints): routes with fewer than 2 waypoints get xref = ones (the first stop
// test of EVAL.m:47,64 then ends them before any iteration) and launch_mark_no_route sets their status afterwards.
cudaError_t launch_resample_routes(int B, int W, int H, int nj, double dt, const double *routes /*nj x W x B*/,
                                   const int *route_len, double *theta0, double *thetag, double *xref, cudaStream_t s);
cudaError_t launch_mark_no_route(int B, const int *route_len, int *status, int *iters, cudaStream_t s);
// route_len_or_fail[s] = fail[s] || route_len[s] < 0 ? 0 : route_len[s]
cudaError_t launch_route_len_or_fail(int S, const int *route_len, const int *fail, int *out, cudaStream_t s);

// C = alpha * op(A) * B  (column-major, A is M x K with lda (or K x M if transA), B is K x N, C is M x N)
cudaError_t launch_dgemm(int M, int N, int K, double alpha, const double *A, int lda, bool transA, const double *B,
                         int ldb, double *C, int ldc, cudaStream_t s);

// ---- per-batch init + the QP / rollout kernel ----------------------------------------------------------------
struct SolveArgs {
  const DevTables *tab;
  int B, H, nj, n, nobs, nprim;  // nprim = 3n
  int solver;                    // 0 CFS, 1 PSGCFS
  int max_outer;
  double eps_outer, alpha;
  int has_lim, has_bounds, margin_is_D;
  const double *G, *gdiag;       // Gram operator used by the QP (QQ metric for CFS, identity metric for PSGCFS)
  const double *QQ;              // n x n as given by the caller (PSGCFS gradient QQ*u, PSGCFS_FANUC.m:131)
  const double *lim, *max_input;
  // per problem inputs
  const double *x0, *ff, *caug, *xref, *noise;
  // per problem state
  double *u0;     // n x B   unconstrained minimiser (CFS) / PSG point (PSGCFS)
  double *v0;     // 3n x B  P*u0
  double *cost0;  // B       cost at u0 (CFS)
  double *fupper; // B       upper bound of the cost over the box |u| <= MAX_input (infeasibility certificate)
  double qq_norm_inf;
  double *u, *x;  // current iterate
  double *dist, *grad;  // K1 outputs: [prob][obs][i], [prob][obs][i][nj]
  double *cost_hist, *e_u_hist;
  int *iters, *status, *flags;
  // scheduling
  int *list_cur, *list_next;  // active problem lists
  int *count_cur, *count_next;
  int *work_counter;          // persistent-CTA work queue
  double *slab;               // per-CTA workspace for the working-set inverse, slab_ld*slab_ld doubles each
  int slab_ld;
  int outer_iter;             // 1-based iteration being executed
  long long *qp_steps;        // device counter
  int *max_active;            // device max
  int *prob_steps;            // per-problem step counter (B)
  // PSGCFS state (solver == 1)
  double *w;                  // n x B   QQ*u of the current iterate (batched GEMM after every projection)
  double *cost_old, *cost_new;  // B     EVAL.cost_old / cost_new (EVAL.m:29, PSGCFS_FANUC.m:66,76,90)
  int *skip;                  // B       stop_inner() was already true: no PSG step this outer iteration (PSGCFS_FANUC.m:88,136-142)
  // fused kernel tiers (k_fused.cu)
  const int *order;           // bulk tier: problem of work-queue slot k (nullptr: slot k = problem k)
  int tier;                   // 0 bulk (all B problems), 1 heavy (the escalation list)
  int *esc_list, *esc_count;  // problems the bulk tier handed over (working set outgrew shared memory / step cap)
  int *work_counter2;         // work queue of the heavy tier
  int esc_steps;              // bulk tier: dual steps per QP before escalation
  long long *prof;            // optional 8-slot phase profile of k_qp (clock64 ticks of thread 0), or nullptr
  // warp-per-problem bulk tier (k_warp.cu)
  double *zslab;              // per-warp overflow of the direction cache: (WQ_QZ - warp_zs) * n doubles per resident warp
  int warp_zs;                // direction slots kept in shared memory
  int warp_qcap;              // working-set capacity of the warp tier (rows), <= 31; beyond it -> heavy tier
  // phase 0 / 1: fresh problems (all B).  phase 2: resume the problems of cont_list (state in x / u / iters / touch) from their
  // next outer iteration.  How far a launch goes is set by it_stop below.
  int phase;
  int one_shot;               // warp tier: grid = one warp per problem, no work queue (CTAs leave the SM after one problem)
  int *cont_list, *cont_count;
  int *touch;                 // B: CFS_FLAG_TOUCH of the problems in cont_list
  // a launch with it_stop > 0 stops every problem after outer iteration it_stop and appends the unfinished ones to cont_out
  // (screening passes: the long dual chains of the early iterations reach the heavy tier while the bulk of the work is
  // still ahead); it_stop = 0: run to the stop rule
  int it_stop;
  int *cont_out, *cont_out_count;
  // per-waypoint margin offsets [prob][obs][i] (same layout as dist), finite and >= 0, or nullptr: the obstacle row of (j, i)
  // uses dist - (margin_j + off) instead of dist - margin_j.  Read only by the instantiations compiled with the offset flag (the
  // launch wrappers pick them when margin_off != nullptr), so the kernels launched without offsets are unchanged.  Last member:
  // the parameter offsets of every other field stay where they were.
  const double *margin_off;
  // joint position limits [qmax (nj) | qmin (nj)] on the device, +-inf for a side without a limit, or nullptr: every QP gets the
  // rows theta_(i+1),k <= qmax_k and -theta_(i+1),k <= -qmin_k (ids OH + 4n + 2e + neg, e = i nj + k; DESIGN.md section 3d).
  // Read only by the limit instantiations, which are also margin-offset instantiations: the launch wrappers require margin_off
  // (a zero buffer when the solve has no offsets) whenever qlim is set.  Last member, like margin_off.
  const double *qlim;
};
cudaError_t launch_solve_init(const SolveArgs &a, cudaStream_t s);
cudaError_t launch_v0(const SolveArgs &a, cudaStream_t s);
// ---- CHOMP_FANUC (k_chomp.cu) ------------------------------------------------------------------------------
struct ChompArgs {
  int B, n, nj, H, nobs, max_outer, it;
  double alpha;
  const DevTables *tab;
  const double *x0, *ff, *caug;  // 2nj x B, n x B, B
  double *u, *x;                 // n x B, 2n x B: the iterate, updated in place
  const double *w;               // QQ * u of the current u (n x B)
  const double *dist, *grad, *linkdist;  // K1d (dm_f mode) at the current x: [b][obstacle][waypoint] (, [joint] / [link])
  double *cost_hist, *e_u_hist;  // max_outer x B
};
cudaError_t launch_chomp_step(const ChompArgs &a, cudaStream_t s);
cudaError_t launch_chomp_cost(const ChompArgs &a, cudaStream_t s);

cudaError_t launch_psg_point(const SolveArgs &a, cudaStream_t s);  // K5: PSG_update_arm point + v0 = P*point
cudaError_t launch_psg_cost(const SolveArgs &a, cudaStream_t s);   // EVAL.get_cost of the projected iterate
cudaError_t launch_qp(const SolveArgs &a, int grid, cudaStream_t s);
size_t qp_smem_bytes(const SolveArgs &a);
int qp_max_grid(const SolveArgs &a, int device);
cudaError_t launch_finalize(const SolveArgs &a, cudaStream_t s);

// ---- fused persistent solver: the whole CFS outer loop of a problem inside one CTA (k_fused.cu) -------------------------
bool fused_supported(const SolveArgs &a);  // CFS solver, num_jac gradients, nj in {2, 5}
size_t fused_smem_bytes(const SolveArgs &a, int tier);
int fused_max_grid(const SolveArgs &a, int device, int tier);
cudaError_t launch_fused(const SolveArgs &a, int grid, int tier, cudaStream_t s);

// ---- warp-per-problem bulk tier of the fused solver (k_warp.cu): cfg 0 = 12 warps in one CTA per SM, 1 = 3 CTAs x 3 warps ----
bool warp_supported(const SolveArgs &a, int cfg);  // CFS solver, num_jac gradients, nj in {2, 5}, shared memory fits
size_t warp_smem_bytes(const SolveArgs &a, int cfg);
int warp_max_grid(const SolveArgs &a, int device, int cfg);
int warp_warps_per_cta(int cfg);
size_t warp_slab_bytes_per_warp(const SolveArgs &a);
// lock-step form of the warp QP (PSGCFS / DERIVEST paths): one outer iteration of list_cur; escalations go to esc_list
bool qp_warp_supported(const SolveArgs &a);
int qp_warp_max_grid(const SolveArgs &a, int device);
cudaError_t launch_qp_warp(const SolveArgs &a, int grid, cudaStream_t s);
cudaError_t launch_warp(const SolveArgs &a, int grid, int cfg, cudaStream_t s);

// ---- dense get_con rows (one problem) -------------------------------------------------------------------------
cudaError_t launch_get_con_rows(const DevTables *tab, int H, int nj, int nobs, int has_lim, int margin_is_D,
                                const double *x0, const double *u, const double *lim, const double *dist,
                                const double *grad, double *Ainq, double *binq, int m, cudaStream_t s);

// ---- FP64 peak micro-benchmark ----------------------------------------------------------------------------------
cudaError_t launch_fp64_peak(double *sink, int iters, int grid, int block, cudaStream_t s);

}  // namespace cfs
