// cfs_api.cu -- C ABI of libcfs_b200.so (include/cfs_b200.h): context, device buffers, stream orchestration.
//
// Host side of the hot path: replaces the bodies of CFS_FANUC.optimizer (Lib/CFS_FANUC.m:62-79) and
// PSGCFS_FANUC.optimizer (Lib/PSGCFS_FANUC.m:65-82) by a fixed, sync-free sequence of kernel launches on one stream:
//   set-up (once per cost):  Cholesky + primitive solve + Gram GEMM                       (k_setup.cu)
//   per batch:               u0 = -QQ^{-1} FF (GEMM), v0 = P u0, init / first stop test   (k_qp.cu)
//   per outer iteration:     K1 distance+gradient over the active list -> K3 QP/roll-out/stop (device work queue,
//                            device-built next active list; the host never reads anything back until the end)
// There is no CPU fallback: every entry point needs a CUDA device.
#include "../../include/cfs_b200.h"

#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <string>
#include <thread>
#include <vector>

#include <nvtx3/nvToolsExt.h>  // header-only NVTX v3: ranges around set-up, copies and the solver tiers (SURVEY.md section 5)

#include "cfs_kernels.cuh"

using namespace cfs;

static thread_local std::string g_create_error;  // last cfs_create failure of the calling thread

struct NvtxRange {
  explicit NvtxRange(const char *name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
};

struct DevBuf {
  void *p = nullptr;
  size_t cap = 0;
};

struct cfs_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;      // stream in use
  cudaStream_t own_stream = nullptr;  // created by cfs_create
  cudaStream_t heavy_stream = nullptr;  // highest priority: the heavy tier must not queue behind other contexts' bulk tiers
  cudaEvent_t ev_bulk = nullptr, ev_heavy = nullptr;
#define CFS_MAX_SCREEN 3
  cudaStream_t heavy_streams[CFS_MAX_SCREEN] = {nullptr, nullptr, nullptr};  // the heavy launches of the screening passes (= heavy_stream)
  cudaEvent_t ev_pass[CFS_MAX_SCREEN] = {nullptr, nullptr, nullptr}, ev_hdone[CFS_MAX_SCREEN] = {nullptr, nullptr, nullptr};
  std::string err;
  // tables
  DevTables htab;
  DevTables *dtab = nullptr;
  DerivestTab *ddv = nullptr;
  bool have_robot = false, have_obs = false, have_cost = false;
  int nj = 0, nobs = 0;
  double motion_R[CFS_MAXL] = {0};  // per-joint motion bound of the continuous checks (cfs_set_robot); kernel argument, not in DevTables
  // cost
  int H = 0, n = 0;
  bool has_lim = false, has_bounds = false;
  // joint position limits (cfs_set_joint_limits): [qmax | qmin] (CFS_MAXL each) on the host and the device
  bool has_qlim = false;
  double hqlim[2 * CFS_MAXL] = {0};
  double *dqlim = nullptr;
  double qq_norm_inf = 0.0;
  double *dQQraw = nullptr;  // QQ exactly as given (PSGCFS gradient); dQQ holds (QQ+QQ')/2
  double *dQQ = nullptr, *dG = nullptr, *dgn = nullptr, *dGI = nullptr, *dgnI = nullptr;
  double *dlim = nullptr, *dumax = nullptr, *dworkL = nullptr, *dworkY = nullptr;
  int *dinfo = nullptr;
  bool have_GI = false;
  // cost blocks for the device-side problem builder (cfs_set_cost_blocks)
  bool have_blocks = false;
  double *dQblk = nullptr;
  double stage_w = 0.0, term_w = 0.0;
  DevBuf th0, thg;
  // batch buffers
  DevBuf x0, ff, caug, xref, noise, u, x, cost, eu, u0, v0, cost0, dist, grad, lid, iters, status, flags, listA, listB,
      counters, slab, scratch_out, qpsteps, fupper, probsteps, psg_w, psg_cost, psg_skip, routes, zslab, cont, rlen,
      chk_out, chk_seg, chk_ctr, rep_off, rep_offo, rep_in, rep_out, rep_list, zero_off;
  DevBuf area;  // the regions of the synchronous host-pointer entries (Area)
  int slab_grid = 0, slab_ld = 0;
  // pinned staging of the host-pointer entries: pageable caller buffers (MATLAB's mxGetPr memory, numpy arrays) are copied
  // through these so that cudaMemcpyAsync stays asynchronous; pinned / registered caller buffers are used in place
  void *stage_in = nullptr, *stage_out = nullptr;
  size_t stage_in_cap = 0, stage_out_cap = 0;
  struct CopyBack { void *dst; const void *src; size_t bytes; };
  std::vector<CopyBack> copy_back;  // staged results to hand to the caller in cfs_wait
  // timing
  std::vector<cudaEvent_t> ev;
  cudaEvent_t ev_a = nullptr, ev_b = nullptr;
  cudaEvent_t ev_h[4] = {nullptr, nullptr, nullptr, nullptr};  // H2D begin/end, D2H begin/end of the host-pointer entry
  struct {
    bool active = false, host = false;
    int B = 0, max_outer = 0;
    const int *d_iters = nullptr, *d_status = nullptr;
  } pending;
  int timing_level = 1;
  bool use_fused = true;  // cfs_set_option("fused")
  int esc_steps = 48;     // cfs_set_option("esc_steps")
  int heavy_grid = 48;    // cfs_set_option("heavy_grid"): cap of the heavy tier's grid (0 = one CTA per SM)
  int bulk_grid = 0;      // cfs_set_option("bulk_grid"): cap of the bulk tier's grid (0 = every resident slot)
  int heavy_prio = 1;     // cfs_set_option("heavy_prio"): heavy tier on the highest-priority stream
  int lpt = 1;            // cfs_set_option("lpt"): fused solver pulls the problems longest-expected-first
  int use_warp = 1;       // cfs_set_option("warp"): bulk tier = one warp per problem (k_warp.cu); 0 = one CTA per problem
  int warp_cfg = 3;       // cfs_set_option("warp_cfg"): CTA shape of the warp tier (k_warp.cu): 0 = 12 warps x 1 CTA/SM, 1 = 3 x 3, 2 = 4 x 3,
                          // 3 = 1 warp x 10 CTAs/SM (default: the finest granularity pipelines best across contexts), 4 = 2 x 5
  int warp_zs = 0;        // cfs_set_option("warp_zs"): direction slots in shared memory (0 = as many as fit, at most 4)
  int use_warp_lockstep = 0;  // cfs_set_option("warp_lockstep"): launch-per-iteration path solves its QPs with k_qp_warp (measured: no gain --
                              // a lock-step iteration still waits for its slowest QP, and that one is slower on a single warp)
  int one_shot = 0;       // cfs_set_option("one_shot"): warp tier without a work queue, one problem per warp
  long long last_warp_grid_warps = 0, last_sms = 0;  // cfs_get_warp_profile
  int screen = 2;         // cfs_set_option("screen"): number of screening passes (0..3): outer iterations 1..screen of the warp tier in launches of their own, each followed by a heavy launch
  long long warp_key = -1;  // cache of the warp tier's launch configuration
  int warp_zs_pick = 0, warp_grid_pick = 0;
  int warp_qcap = 15;     // cfs_set_option("warp_qcap"): working-set rows the warp tier keeps (<= 31; inverse + directions spill to L2 beyond 16:
                          // measured, a single warp on a 16..31-row working set lengthens the tail more than the heavy tier costs)
  int heavy_cfg = 0;      // cfs_set_option("heavy_cfg"): 0 = 144 x 144 inverse on chip (whole SM), 1 = slim (64 x 64 on chip, 168 registers)
  int heavy_skip = 0;     // cfs_set_option("heavy_skip"): measurement only -- the heavy tier is not launched (escalated problems keep status 4)
  bool fused_last = false;
  std::vector<double> it_grad_ms, it_qp_ms;
  cfs_stats stats;
};

static int fail(cfs_ctx *c, int code, const char *fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  if (c)
    c->err = buf;
  else
    g_create_error = buf;
  return code;
}

#define CU(call)                                                                                     \
  do {                                                                                               \
    cudaError_t e_ = (call);                                                                         \
    if (e_ != cudaSuccess)                                                                           \
      return fail(ctx, CFS_E_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
  } while (0)

static int ensure(cfs_ctx *ctx, DevBuf &b, size_t bytes) {
  if (bytes <= b.cap) return 0;
  if (b.p) cudaFree(b.p);
  b.p = nullptr;
  b.cap = 0;
  cudaError_t e = cudaMalloc(&b.p, bytes);
  if (e != cudaSuccess) return fail(ctx, CFS_E_NOMEM, "cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
  b.cap = bytes;
  return 0;
}
template <class T>
static T *ptr(DevBuf &b) {
  return reinterpret_cast<T *>(b.p);
}

extern "C" const char *cfs_version(void) { return "cfs_b200 0.1 (sm_100a)"; }

extern "C" const char *cfs_last_error(const cfs_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

extern "C" int cfs_create(cfs_ctx **out, int device_id) {
  if (!out) return fail(nullptr, CFS_E_ARG, "cfs_create: out is NULL");
  *out = nullptr;
  // Several contexts pipeline copy | solve | copy on their own streams; with the default of 8 hardware queues the copies of
  // one context queue behind the persistent kernels of another: hosts that run more than 8 contexts should export
  // CUDA_DEVICE_MAX_CONNECTIONS=32 before their first CUDA call (bench.py and the MEX loader do; INTEGRATION.md).  The library
  // never touches the process environment.
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(nullptr, CFS_E_CUDA, "cfs_create: no CUDA device (%s); libcfs_b200 has no CPU fallback",
                cudaGetErrorString(e));
  if (device_id < 0 || device_id >= ndev) return fail(nullptr, CFS_E_ARG, "cfs_create: device %d of %d", device_id, ndev);
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, device_id);
  if (prop.major != 10)
    return fail(nullptr, CFS_E_CUDA, "cfs_create: device %d is sm_%d%d; this library is built for sm_100a only", device_id,
                prop.major, prop.minor);
  cfs_ctx *ctx = new cfs_ctx();
  ctx->device = device_id;
  memset(&ctx->stats, 0, sizeof(ctx->stats));
  memset(&ctx->htab, 0, sizeof(ctx->htab));
  if (cudaSetDevice(device_id) != cudaSuccess || cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaMalloc(&ctx->dtab, sizeof(DevTables)) != cudaSuccess || cudaMalloc(&ctx->ddv, sizeof(DerivestTab)) != cudaSuccess ||
      cudaMalloc(&ctx->dinfo, sizeof(int)) != cudaSuccess || cudaEventCreate(&ctx->ev_a) != cudaSuccess ||
      cudaEventCreate(&ctx->ev_b) != cudaSuccess) {
    fail(nullptr, CFS_E_CUDA, "cfs_create: %s", cudaGetErrorString(cudaGetLastError()));
    delete ctx;
    return CFS_E_CUDA;
  }
  // DERIVEST constants (derivest.m:203,238,282,431,493-525), FP64 on the host once
  DerivestTab dv;
  memset(&dv, 0, sizeof(dv));
  {
    const double sr = 2.0000001, srinv = 1.0 / sr;
    for (int k = 0; k < DV_NDEL; ++k) dv.delta[k] = 100.0 * pow(sr, (double)(-k));
    // fdarule = [1 0]/fdamat(sr,1,2), fdamat(i,j)=c(j)*srinv^((i-1)(2j-1)), c=[1 1/6]
    double A[2][3] = {{1.0, srinv, 1.0}, {1.0 / 6.0, (1.0 / 6.0) * pow(srinv, 3), 0.0}};
    if (fabs(A[1][0]) > fabs(A[0][0]))
      for (int k = 0; k < 3; ++k) std::swap(A[0][k], A[1][k]);
    const double f = A[1][0] / A[0][0];
    A[1][1] -= f * A[0][1];
    A[1][2] -= f * A[0][2];
    dv.fdarule[1] = A[1][2] / A[1][1];
    dv.fdarule[0] = (A[0][2] - A[0][1] * dv.fdarule[1]) / A[0][0];
    const double ex[2] = {4, 6};
    for (int i = 0; i < 4; ++i) {
      dv.rmat[i][0] = 1.0;
      for (int j = 0; j < 2; ++j) dv.rmat[i][1 + j] = (i == 0) ? 1.0 : pow(srinv, i * ex[j]);
    }
    for (int j = 0; j < 3; ++j) {  // economy QR by twice-iterated modified Gram-Schmidt
      double v[4];
      for (int i = 0; i < 4; ++i) v[i] = dv.rmat[i][j];
      for (int k = 0; k < 3; ++k) dv.rr[k][j] = 0;
      for (int pass = 0; pass < 2; ++pass)
        for (int k = 0; k < j; ++k) {
          double dot = 0;
          for (int i = 0; i < 4; ++i) dot += dv.q[i][k] * v[i];
          dv.rr[k][j] += dot;
          for (int i = 0; i < 4; ++i) v[i] -= dot * dv.q[i][k];
        }
      double nn = 0;
      for (int i = 0; i < 4; ++i) nn += v[i] * v[i];
      nn = sqrt(nn);
      dv.rr[j][j] = nn;
      for (int i = 0; i < 4; ++i) dv.q[i][j] = v[i] / nn;
    }
    double rinv[3][3] = {{0}};
    for (int c = 0; c < 3; ++c)
      for (int i = 2; i >= 0; --i) {
        double s = (i == c) ? 1.0 : 0.0;
        for (int k = i + 1; k < 3; ++k) s -= dv.rr[i][k] * rinv[k][c];
        rinv[i][c] = s / dv.rr[i][i];
      }
    const double cov11 = rinv[0][0] * rinv[0][0] + rinv[0][1] * rinv[0][1] + rinv[0][2] * rinv[0][2];
    dv.errfac = 12.7062047361747 * sqrt(cov11);
  }
  cudaMemcpy(ctx->ddv, &dv, sizeof(dv), cudaMemcpyHostToDevice);
  ctx->own_stream = ctx->stream;
  {
    int lo = 0, hi = 0;
    cudaDeviceGetStreamPriorityRange(&lo, &hi);  // hi is the numerically lowest = highest priority
    if (cudaStreamCreateWithPriority(&ctx->heavy_stream, cudaStreamNonBlocking, hi) != cudaSuccess) ctx->heavy_stream = nullptr;
    cudaEventCreate(&ctx->ev_bulk);   // timing enabled: cfs_dev_timeline
    cudaEventCreate(&ctx->ev_heavy);
    ctx->heavy_streams[0] = ctx->heavy_stream;
    for (int p = 0; p < CFS_MAX_SCREEN; ++p) {
      ctx->heavy_streams[p] = ctx->heavy_stream;  // one heavy stream per context: streams beyond the device's hardware queues
                                                  // (CUDA_DEVICE_MAX_CONNECTIONS <= 32) only buy false dependencies
      cudaEventCreate(&ctx->ev_pass[p]);
      cudaEventCreate(&ctx->ev_hdone[p]);
    }
  }
  *out = ctx;
  return 0;
}

extern "C" int cfs_set_stream(cfs_ctx *ctx, void *cuda_stream) {
  if (!ctx) return CFS_E_ARG;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  ctx->stream = cuda_stream ? reinterpret_cast<cudaStream_t>(cuda_stream) : ctx->own_stream;
  return 0;
}

static void free_buf(DevBuf &b) {
  if (b.p) cudaFree(b.p);
  b.p = nullptr;
  b.cap = 0;
}

extern "C" void cfs_destroy(cfs_ctx *ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  DevBuf *bufs[] = {&ctx->x0, &ctx->ff, &ctx->caug, &ctx->xref, &ctx->noise, &ctx->u, &ctx->x, &ctx->cost, &ctx->eu,
                    &ctx->u0, &ctx->v0, &ctx->cost0, &ctx->dist, &ctx->grad, &ctx->lid, &ctx->iters, &ctx->status,
                    &ctx->flags, &ctx->listA, &ctx->listB, &ctx->counters, &ctx->slab,
                    &ctx->scratch_out, &ctx->qpsteps, &ctx->fupper, &ctx->probsteps, &ctx->routes, &ctx->psg_w, &ctx->psg_cost,
                    &ctx->psg_skip, &ctx->th0, &ctx->thg, &ctx->zslab, &ctx->cont, &ctx->rlen,
                    &ctx->chk_out, &ctx->chk_seg, &ctx->chk_ctr, &ctx->rep_off, &ctx->rep_offo, &ctx->rep_in,
                    &ctx->rep_out, &ctx->rep_list, &ctx->zero_off, &ctx->area};
  for (DevBuf *b : bufs) free_buf(*b);
  if (ctx->dQblk) cudaFree(ctx->dQblk);
  if (ctx->dqlim) cudaFree(ctx->dqlim);
  double *ds[] = {ctx->dQQraw, ctx->dQQ, ctx->dG, ctx->dgn, ctx->dGI, ctx->dgnI, ctx->dlim, ctx->dumax, ctx->dworkL, ctx->dworkY};
  for (double *d : ds)
    if (d) cudaFree(d);
  if (ctx->dtab) cudaFree(ctx->dtab);
  if (ctx->ddv) cudaFree(ctx->ddv);
  if (ctx->dinfo) cudaFree(ctx->dinfo);
  for (cudaEvent_t e : ctx->ev) cudaEventDestroy(e);
  if (ctx->ev_a) cudaEventDestroy(ctx->ev_a);
  if (ctx->ev_b) cudaEventDestroy(ctx->ev_b);
  for (cudaEvent_t e : ctx->ev_h)
    if (e) cudaEventDestroy(e);
  if (ctx->stage_in) cudaFreeHost(ctx->stage_in);
  if (ctx->stage_out) cudaFreeHost(ctx->stage_out);
  if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
  if (ctx->heavy_stream) cudaStreamDestroy(ctx->heavy_stream);
  if (ctx->ev_bulk) cudaEventDestroy(ctx->ev_bulk);
  if (ctx->ev_heavy) cudaEventDestroy(ctx->ev_heavy);
  for (int p = 0; p < CFS_MAX_SCREEN; ++p) {
    if (ctx->ev_pass[p]) cudaEventDestroy(ctx->ev_pass[p]);
    if (ctx->ev_hdone[p]) cudaEventDestroy(ctx->ev_hdone[p]);
  }
  delete ctx;
}

static int upload_tables(cfs_ctx *ctx) {
  CU(cudaSetDevice(ctx->device));
  CU(cudaMemcpyAsync(ctx->dtab, &ctx->htab, sizeof(DevTables), cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return 0;
}

// Motion bound of the continuous checks: R[j] >= ||dp/dtheta_j|| for every link-axis endpoint p of the links l >= j, at every
// theta.  Joint j turns everything downstream of it about an axis through its frame origin: the own translation contributes its
// rotating part a_j (the constant part -- d_j along the axis, or robot.T on the 2L arm -- does not move), every later link at most
// |a_i| + |(tx_i, ty_i, dz_i)|, the endpoint itself |cap|.  Triangle inequality; the same sums in the same order as
// orc_motion_bound (tests/check_oracle.c).
static void motion_bound(const DevTables &t, int nj, double R[CFS_MAXL]) {
  for (int j = 0; j < CFS_MAXL; ++j) R[j] = 0.0;
  for (int j = 0; j < nj; ++j) {
    double reach = fabs(t.link[j].a);
    for (int l = j; l < nj; ++l) {
      const LinkTab &L = t.link[l];
      if (l > j) reach = reach + (fabs(L.a) + sqrt((L.tx * L.tx + L.ty * L.ty) + L.dz * L.dz));
      for (int k = 0; k < 2; ++k) {
        const double c = sqrt((L.cap[k][0] * L.cap[k][0] + L.cap[k][1] * L.cap[k][1]) + L.cap[k][2] * L.cap[k][2]);
        if (reach + c > R[j]) R[j] = reach + c;
      }
    }
  }
}

extern "C" int cfs_set_robot(cfs_ctx *ctx, int robot_kind, const double *DH, int dh_rows, const double *base,
                             const double *cap_p, int n_joints, const double *T2L, double dt) {
  if (!ctx) return CFS_E_ARG;
  if (!DH || !base || !cap_p) return fail(ctx, CFS_E_ARG, "cfs_set_robot: NULL argument");
  if (n_joints < 2 || n_joints > CFS_MAXL || dh_rows < n_joints)
    return fail(ctx, CFS_E_ARG, "cfs_set_robot: n_joints=%d (2..%d), dh_rows=%d", n_joints, CFS_MAXL, dh_rows);
  if (robot_kind < CFS_ROBOT_M16IB || robot_kind > CFS_ROBOT_2L) return fail(ctx, CFS_E_ARG, "cfs_set_robot: kind %d", robot_kind);
  if (robot_kind == CFS_ROBOT_2L && !T2L) return fail(ctx, CFS_E_ARG, "cfs_set_robot: 2L needs robot.T");
  if (!(dt > 0)) return fail(ctx, CFS_E_ARG, "cfs_set_robot: dt must be positive");
  DevTables &t = ctx->htab;
  for (int i = 0; i < CFS_MAXL; ++i) memset(&t.link[i], 0, sizeof(LinkTab));
  for (int i = 0; i < n_joints; ++i) {
    LinkTab &L = t.link[i];
    const double d = DH[i + dh_rows * 1], a = DH[i + dh_rows * 2], al = DH[i + dh_rows * 3];
    if (robot_kind == CFS_ROBOT_2L) {  // CapPos2.m:21-27: R = Rz(theta), T = robot.T(:,i+1)
      L.ca = 1.0;
      L.sa = 0.0;
      L.a = 0.0;
      L.tx = T2L[0 + 3 * (i + 1 < 3 ? i + 1 : 2)];
      L.ty = T2L[1 + 3 * (i + 1 < 3 ? i + 1 : 2)];
      L.dz = T2L[2 + 3 * (i + 1 < 3 ? i + 1 : 2)];
    } else {  // CapPos.m:13-16
      L.ca = cos(al);
      L.sa = sin(al);
      L.a = a;
      L.tx = 0.0;
      L.ty = 0.0;
      L.dz = d;
    }
    L.th_off = (robot_kind == CFS_ROBOT_M200I && i == 1) ? -(3.14159265358979323846 / 2) : 0.0;  // dist_arm_3D_200i_2.m:11
    for (int k = 0; k < 2; ++k)
      for (int c = 0; c < 3; ++c) L.cap[k][c] = cap_p[c + 3 * k + 6 * i];
  }
  for (int c = 0; c < 3; ++c) t.base[c] = base[c];
  t.dt = dt;
  t.kind = robot_kind;
  t.nj = n_joints;
  motion_bound(t, n_joints, ctx->motion_R);
  ctx->nj = n_joints;
  ctx->has_qlim = false;  // nj may change
  for (double &v : ctx->hqlim) v = 0.0;
  ctx->have_robot = true;
  ctx->have_cost = false;  // n depends on nj
  return upload_tables(ctx);
}

extern "C" int cfs_set_obstacles_ex(cfs_ctx *ctx, const double *seg, const int *kind, const double *D, const double *eps, int n_obs) {
  if (!ctx) return CFS_E_ARG;
  if (n_obs < 0 || n_obs > CFS_MAX_OBS) return fail(ctx, CFS_E_ARG, "cfs_set_obstacles: n_obs=%d (0..%d)", n_obs, CFS_MAX_OBS);
  if (n_obs > 0 && !seg) return fail(ctx, CFS_E_ARG, "cfs_set_obstacles: NULL seg");
  DevTables &t = ctx->htab;
  for (int j = 0; j < n_obs; ++j) {
    ObsTab &o = t.obs[j];
    memset(&o, 0, sizeof(o));
    const int kd = kind ? kind[j] : CFS_OBS_CAPSULE;
    if (kd != CFS_OBS_CAPSULE && kd != CFS_OBS_BOX) return fail(ctx, CFS_E_ARG, "cfs_set_obstacles: obstacle %d has kind %d", j, kd);
    o.kind = kd;
    o.D = D ? D[j] : 0.0;
    o.eps = eps ? eps[j] : 0.0;
    if (kd == CFS_OBS_BOX) {  // seg = [min corner, max corner]
      for (int c = 0; c < 3; ++c) {
        o.s[c] = seg[c + 6 * j];
        o.d2[c] = seg[3 + c + 6 * j];
        if (!(o.s[c] <= o.d2[c])) return fail(ctx, CFS_E_ARG, "cfs_set_obstacles: box %d has min > max on axis %d", j, c);
      }
      continue;
    }
    double D2 = 0.0;
    for (int c = 0; c < 3; ++c) {
      o.s[c] = seg[c + 6 * j];
      o.d2[c] = seg[3 + c + 6 * j] - seg[c + 6 * j];  // distLinSeg.m:26
    }
    for (int c = 0; c < 3; ++c) D2 += o.d2[c] * o.d2[c];  // distLinSeg.m:30
    o.D2 = D2;
    o.rD2 = D2 != 0.0 ? 1.0 / D2 : 0.0;
  }
  t.nobs = n_obs;
  ctx->nobs = n_obs;
  ctx->have_obs = true;
  return upload_tables(ctx);
}

extern "C" int cfs_set_obstacles(cfs_ctx *ctx, const double *seg, const double *D, const double *eps, int n_obs) {
  return cfs_set_obstacles_ex(ctx, seg, nullptr, D, eps, n_obs);
}

extern "C" int cfs_set_joint_limits(cfs_ctx *ctx, const double *qmin, const double *qmax) {
  if (!ctx) return CFS_E_ARG;
  if (!ctx->have_robot) return fail(ctx, CFS_E_STATE, "cfs_set_joint_limits: call cfs_set_robot first");
  if (!qmin != !qmax) return fail(ctx, CFS_E_ARG, "cfs_set_joint_limits: qmin and qmax must both be given or both be NULL");
  const int nj = ctx->nj;
  if (!qmin) {
    ctx->has_qlim = false;
    for (double &v : ctx->hqlim) v = 0.0;
    return 0;
  }
  for (int k = 0; k < nj; ++k)
    if (qmin[k] != qmin[k] || qmax[k] != qmax[k] || !(qmin[k] <= qmax[k]) || qmin[k] == INFINITY || qmax[k] == -INFINITY)
      return fail(ctx, CFS_E_ARG, "cfs_set_joint_limits: joint %d has qmin = %g, qmax = %g", k, qmin[k], qmax[k]);
  CU(cudaSetDevice(ctx->device));
  if (!ctx->dqlim) CU(cudaMalloc(&ctx->dqlim, sizeof(double) * 2 * CFS_MAXL));
  double h[2 * CFS_MAXL] = {0};
  for (int k = 0; k < nj; ++k) {  // the kernels' layout: qmax (nj) | qmin (nj)
    h[k] = qmax[k];
    h[nj + k] = qmin[k];
  }
  CU(cudaMemcpyAsync(ctx->dqlim, h, sizeof(h), cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  for (int k = 0; k < 2 * CFS_MAXL; ++k) ctx->hqlim[k] = h[k];
  ctx->has_qlim = true;
  return 0;
}

extern "C" int cfs_set_cost(cfs_ctx *ctx, int H, const double *QQ, const double *lim, const double *max_input) {
  if (!ctx) return CFS_E_ARG;
  if (!ctx->have_robot) return fail(ctx, CFS_E_STATE, "cfs_set_cost: call cfs_set_robot first");
  if (H < 1 || !QQ) return fail(ctx, CFS_E_ARG, "cfs_set_cost: H=%d", H);
  CU(cudaSetDevice(ctx->device));
  const int nj = ctx->nj, n = H * nj, np = 3 * n;
  double *ds[] = {ctx->dQQraw, ctx->dQQ, ctx->dG, ctx->dgn, ctx->dGI, ctx->dgnI, ctx->dlim, ctx->dumax, ctx->dworkL, ctx->dworkY};
  for (double *d : ds)
    if (d) cudaFree(d);
  ctx->dQQraw = ctx->dQQ = ctx->dG = ctx->dgn = ctx->dGI = ctx->dgnI = ctx->dlim = ctx->dumax = ctx->dworkL = ctx->dworkY = nullptr;
  ctx->have_cost = false;
  ctx->have_GI = false;
  ctx->have_blocks = false;
  CU(cudaMalloc(&ctx->dQQ, sizeof(double) * n * n));
  CU(cudaMalloc(&ctx->dQQraw, sizeof(double) * n * n));
  CU(cudaMemcpyAsync(ctx->dQQraw, QQ, sizeof(double) * n * n, cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMalloc(&ctx->dG, sizeof(double) * (size_t)np * np));
  CU(cudaMalloc(&ctx->dgn, sizeof(double) * np));
  CU(cudaMalloc(&ctx->dworkL, sizeof(double) * n * n));
  CU(cudaMalloc(&ctx->dworkY, sizeof(double) * (size_t)n * np));
  CU(cudaMalloc(&ctx->dlim, sizeof(double) * CFS_MAXL));
  CU(cudaMalloc(&ctx->dumax, sizeof(double) * n));
  // symmetrise on the host: quadprog uses (QQ+QQ')/2 semantics for the quadratic form
  std::vector<double> q((size_t)n * n);
  for (int i = 0; i < n; ++i)
    for (int j = 0; j < n; ++j) q[i + (size_t)n * j] = 0.5 * (QQ[i + (size_t)n * j] + QQ[j + (size_t)n * i]);
  ctx->qq_norm_inf = 0.0;
  for (int i = 0; i < n; ++i) {
    double rs = 0.0;
    for (int j = 0; j < n; ++j) rs += fabs(q[i + (size_t)n * j]);
    if (rs > ctx->qq_norm_inf) ctx->qq_norm_inf = rs;
  }
  CU(cudaMemcpyAsync(ctx->dQQ, q.data(), sizeof(double) * n * n, cudaMemcpyHostToDevice, ctx->stream));
  double limb[CFS_MAXL] = {0};
  if (lim)
    for (int k = 0; k < nj; ++k) limb[k] = lim[k];
  CU(cudaMemcpyAsync(ctx->dlim, limb, sizeof(limb), cudaMemcpyHostToDevice, ctx->stream));
  if (max_input) CU(cudaMemcpyAsync(ctx->dumax, max_input, sizeof(double) * n, cudaMemcpyHostToDevice, ctx->stream));
  ctx->has_lim = lim != nullptr;
  ctx->has_bounds = max_input != nullptr;
  NvtxRange nvtx_setup("cfs:set_cost (Cholesky + Gram operator)");
  CU(cudaEventRecord(ctx->ev_a, ctx->stream));
  CU(setup_gram(n, H, nj, ctx->htab.dt, ctx->dQQ, ctx->dworkL, ctx->dworkY, ctx->dG, ctx->dgn, ctx->dinfo, ctx->stream));
  CU(cudaEventRecord(ctx->ev_b, ctx->stream));
  int info = 0;
  CU(cudaMemcpyAsync(&info, ctx->dinfo, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  float ms = 0;
  cudaEventElapsedTime(&ms, ctx->ev_a, ctx->ev_b);
  ctx->stats.ms_setup = ms;
  if (info != 0) return fail(ctx, CFS_E_NUMERIC, "cfs_set_cost: QQ is not positive definite (pivot %d)", info);
  ctx->H = H;
  ctx->n = n;
  ctx->have_cost = true;
  return 0;
}

extern "C" int cfs_set_cost_blocks(cfs_ctx *ctx, int H, const double *Q, const double *Rblk, double r_scale,
                                   double stage_w, double term_w, const double *lim, const double *max_input) {
  if (!ctx) return CFS_E_ARG;
  if (!ctx->have_robot) return fail(ctx, CFS_E_STATE, "cfs_set_cost_blocks: call cfs_set_robot first");
  if (H < 1 || !Q || !Rblk) return fail(ctx, CFS_E_ARG, "cfs_set_cost_blocks: bad argument");
  CU(cudaSetDevice(ctx->device));
  const int nj = ctx->nj, n = H * nj, ns = 2 * nj;
  if (!ctx->dQblk) CU(cudaMalloc(&ctx->dQblk, sizeof(double) * (4 * CFS_MAXL * CFS_MAXL + CFS_MAXL * CFS_MAXL)));
  double *dR = ctx->dQblk + 4 * CFS_MAXL * CFS_MAXL, *dQQ = nullptr;
  CU(cudaMemcpyAsync(ctx->dQblk, Q, sizeof(double) * ns * ns, cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(dR, Rblk, sizeof(double) * nj * nj, cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMalloc(&dQQ, sizeof(double) * (size_t)n * n));
  cudaError_t e = launch_build_qq(H, nj, ctx->htab.dt, ctx->dQblk, dR, r_scale, stage_w, term_w, dQQ, ctx->stream);
  std::vector<double> qq((size_t)n * n);
  if (e == cudaSuccess) e = cudaMemcpyAsync(qq.data(), dQQ, sizeof(double) * (size_t)n * n, cudaMemcpyDeviceToHost, ctx->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  cudaFree(dQQ);
  if (e != cudaSuccess) return fail(ctx, CFS_E_CUDA, "cfs_set_cost_blocks: %s", cudaGetErrorString(e));
  int rc = cfs_set_cost(ctx, H, qq.data(), lim, max_input);  // symmetrise, factor, Gram operator
  if (rc) return rc;
  ctx->stage_w = stage_w;
  ctx->term_w = term_w;
  ctx->have_blocks = true;
  return 0;
}

static int ensure_GI(cfs_ctx *ctx) {  // identity-metric Gram operator for the PSGCFS projection
  if (ctx->have_GI) return 0;
  const int n = ctx->n, np = 3 * n;
  CU(cudaMalloc(&ctx->dGI, sizeof(double) * (size_t)np * np));
  CU(cudaMalloc(&ctx->dgnI, sizeof(double) * np));
  CU(setup_gram(n, ctx->H, ctx->nj, ctx->htab.dt, nullptr, ctx->dworkL, ctx->dworkY, ctx->dGI, ctx->dgnI, ctx->dinfo,
                ctx->stream));
  ctx->have_GI = true;
  return 0;
}

static int check_ready(cfs_ctx *ctx, bool need_cost) {
  if (!ctx->have_robot) return fail(ctx, CFS_E_STATE, "robot not set (cfs_set_robot)");
  if (!ctx->have_obs) return fail(ctx, CFS_E_STATE, "obstacles not set (cfs_set_obstacles)");
  if (need_cost && !ctx->have_cost) return fail(ctx, CFS_E_STATE, "cost not set (cfs_set_cost)");
  return 0;
}

// The distance/gradient kernel over B trajectories (x: 2n x B, H waypoints each): dist and flags per problem, [b][obstacle][i]
static GradArgs traj_grad_args(const cfs_ctx *ctx, int B, const double *x, double *dist, double *grad, int *flags) {
  GradArgs g;
  memset(&g, 0, sizeof(g));
  g.tab = ctx->dtab; g.dv = ctx->ddv;
  g.x = x; g.ld_prob = 2 * ctx->n; g.ld_i = 2 * ctx->nj;
  g.nslots = B; g.H = ctx->H; g.nj = ctx->nj; g.nobs = ctx->nobs;
  g.o_prob = ctx->nobs * ctx->H; g.o_obs = ctx->H; g.o_i = 1;
  g.dist = dist; g.grad = grad; g.flags = flags;
  return g;
}

// ---- the solve, device pointers --------------------------------------------------------------------------------------
static int solve_device(cfs_ctx *ctx, int B, int solver, int grad, const double *x0, const double *ff,
                        const double *caug, const double *xref, const double *noise, double eps_outer, int max_outer,
                        double alpha, double *u, double *x, double *cost_hist, double *e_u_hist, int *iters, int *status,
                        const double *margin_off = nullptr) {
  const int nj = ctx->nj, H = ctx->H, n = ctx->n, np = 3 * n, O = ctx->nobs, OH = O * H;
  cudaStream_t st = ctx->stream;
  const bool psg = solver == CFS_SOLVER_PSGCFS;
  int rc;
  if (psg) {
    if ((rc = ensure_GI(ctx))) return rc;
    if ((rc = ensure(ctx, ctx->psg_w, sizeof(double) * (size_t)n * B))) return rc;
    if ((rc = ensure(ctx, ctx->psg_cost, sizeof(double) * 2 * B))) return rc;
    if ((rc = ensure(ctx, ctx->psg_skip, sizeof(int) * B))) return rc;
  }
  if ((rc = ensure(ctx, ctx->u0, sizeof(double) * (size_t)n * B))) return rc;
  if ((rc = ensure(ctx, ctx->v0, sizeof(double) * (size_t)np * B))) return rc;
  if ((rc = ensure(ctx, ctx->cost0, sizeof(double) * B))) return rc;
  if ((rc = ensure(ctx, ctx->fupper, sizeof(double) * B))) return rc;
  if ((rc = ensure(ctx, ctx->probsteps, sizeof(int) * B))) return rc;
  if ((rc = ensure(ctx, ctx->dist, sizeof(double) * (size_t)(OH > 0 ? OH : 1) * B))) return rc;
  if ((rc = ensure(ctx, ctx->grad, sizeof(double) * (size_t)(OH > 0 ? OH : 1) * nj * B))) return rc;
  if ((rc = ensure(ctx, ctx->flags, sizeof(int) * B))) return rc;
  if ((rc = ensure(ctx, ctx->listA, sizeof(int) * B))) return rc;
  if ((rc = ensure(ctx, ctx->listB, sizeof(int) * B))) return rc;
  if ((rc = ensure(ctx, ctx->counters, sizeof(int) * 64))) return rc;
  if ((rc = ensure(ctx, ctx->cont, sizeof(int) * 8 * (size_t)B))) return rc;
  if ((rc = ensure(ctx, ctx->qpsteps, sizeof(long long) * 32))) return rc;

  SolveArgs a;
  memset(&a, 0, sizeof(a));
  a.tab = ctx->dtab;
  a.B = B; a.H = H; a.nj = nj; a.n = n; a.nobs = O; a.nprim = np;
  a.solver = solver;
  a.max_outer = max_outer;
  a.eps_outer = eps_outer;
  a.alpha = alpha;
  a.has_lim = ctx->has_lim;
  // PSGCFS: margin obs.D (PSGCFS_FANUC.m:158), projection quadprog(I,-u_,Ainq,binq) without bounds (:120)
  a.has_bounds = psg ? 0 : ctx->has_bounds;
  a.margin_is_D = psg ? 1 : 0;
  a.G = psg ? ctx->dGI : ctx->dG;
  a.gdiag = psg ? ctx->dgnI : ctx->dgn;
  a.QQ = ctx->dQQraw;
  if (psg) {
    a.w = ptr<double>(ctx->psg_w);
    a.cost_old = ptr<double>(ctx->psg_cost);
    a.cost_new = ptr<double>(ctx->psg_cost) + B;
    a.skip = ptr<int>(ctx->psg_skip);
  }
  a.lim = ctx->dlim;
  a.max_input = ctx->dumax;
  a.x0 = x0; a.ff = ff; a.caug = caug; a.xref = xref; a.noise = noise;
  a.u0 = ptr<double>(ctx->u0); a.v0 = ptr<double>(ctx->v0); a.cost0 = ptr<double>(ctx->cost0);
  a.fupper = psg ? nullptr : ptr<double>(ctx->fupper);
  a.qq_norm_inf = ctx->qq_norm_inf;
  a.u = u; a.x = x;
  a.dist = ptr<double>(ctx->dist); a.grad = ptr<double>(ctx->grad);
  a.cost_hist = cost_hist; a.e_u_hist = e_u_hist; a.iters = iters; a.status = status;
  a.flags = ptr<int>(ctx->flags);
  int *cnt = ptr<int>(ctx->counters);  // [0]=count A, [1]=count B, [2]=work counter, [3]=max_active
  a.qp_steps = ptr<long long>(ctx->qpsteps);
  a.max_active = cnt + 3;
  a.prob_steps = ptr<int>(ctx->probsteps);
  a.prof = ctx->timing_level >= 3 ? ptr<long long>(ctx->qpsteps) + 8 : nullptr;
  a.slab_ld = n;
  a.margin_off = O > 0 ? margin_off : nullptr;  // non-null selects the offset instantiations of every solver kernel
  if (ctx->has_qlim) {
    // the joint-limit instantiations are offset instantiations too: without offsets they read zeros, and dist - (m + 0.0)
    // equals dist - m bit for bit
    a.qlim = ctx->dqlim;
    if (!a.margin_off) {
      const size_t ne = (size_t)(OH > 0 ? OH : 1) * B;
      if ((rc = ensure(ctx, ctx->zero_off, sizeof(double) * ne))) return rc;
      CU(cudaMemsetAsync(ctx->zero_off.p, 0, sizeof(double) * ne, st));
      a.margin_off = ptr<double>(ctx->zero_off);
    }
  }

  const bool fused = ctx->use_fused && !psg && grad == CFS_GRAD_NUMJAC && fused_supported(a);
  // bulk tier of the fused solver: one warp per problem (k_warp.cu) when its shared-memory regions fit
  bool warp = false;
  a.warp_qcap = ctx->warp_qcap;
  int warp_grid = 0;
  if (fused && ctx->use_warp) {
    // direction slots in shared memory: the count that keeps the most problems resident per SM (ties: more slots); cached per
    // (n, obstacles, CTA shape)
    const long long key = ((long long)n << 24) ^ ((long long)O << 16) ^ ((long long)ctx->warp_cfg << 8) ^ ctx->warp_zs ^
                          (a.margin_off ? 1LL << 48 : 0) ^  // the offset instantiations have kernel attributes of their own
                          (a.qlim ? 1LL << 49 : 0);         // ... and so have the joint-limit ones
    if (key != ctx->warp_key) {
      ctx->warp_key = key;
      ctx->warp_zs_pick = 0;
      ctx->warp_grid_pick = 0;
      for (int zs = ctx->warp_zs > 0 ? ctx->warp_zs : 4; zs >= 1; --zs) {
        a.warp_zs = zs;
        if (warp_supported(a, ctx->warp_cfg)) {
          const int g = warp_max_grid(a, ctx->device, ctx->warp_cfg);
          if (g > ctx->warp_grid_pick) {
            ctx->warp_grid_pick = g;
            ctx->warp_zs_pick = zs;
          }
        }
        if (ctx->warp_zs > 0) break;
      }
      if (ctx->warp_zs_pick > 0) {  // leave the kernel's dynamic shared-memory limit at the chosen configuration
        a.warp_zs = ctx->warp_zs_pick;
        warp_max_grid(a, ctx->device, ctx->warp_cfg);
      }
    }
    warp = ctx->warp_zs_pick > 0 && ctx->warp_grid_pick > 0;
    a.warp_zs = ctx->warp_zs_pick;
    warp_grid = ctx->warp_grid_pick;
  }
  int grid = fused ? (warp ? warp_grid : fused_max_grid(a, ctx->device, 0)) : qp_max_grid(a, ctx->device);
  const int heavy_tier = ctx->heavy_cfg ? 2 : 1;
  int grid_heavy = fused ? fused_max_grid(a, ctx->device, heavy_tier) : 0;
  if (grid <= 0 || (fused && grid_heavy <= 0))
    return fail(ctx, CFS_E_CUDA, "solver kernel does not fit on this device (shared memory)");
  {
    int sms = 0;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device);
    if (grid > 16 * sms) grid = 16 * sms;
  }
  if (warp) {
    const int wpc = warp_warps_per_cta(ctx->warp_cfg);
    {
      int sms = 0;
      cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device);
      ctx->last_sms = sms;
      ctx->last_warp_grid_warps = (long long)warp_grid * wpc;  // resident warps of a full grid
    }
    a.one_shot = ctx->one_shot;
    if (grid > (B + wpc - 1) / wpc || ctx->one_shot) grid = (B + wpc - 1) / wpc;
    if (grid < 1) grid = 1;
    if ((rc = ensure(ctx, ctx->zslab, warp_slab_bytes_per_warp(a) * (size_t)grid * wpc))) return rc;
    a.zslab = ptr<double>(ctx->zslab);
  }
  if (grid > B) grid = B;
  if (grid < 1) grid = 1;
  if (grid_heavy > B) grid_heavy = B;
  if (fused && ctx->heavy_grid > 0 && grid_heavy > ctx->heavy_grid) grid_heavy = ctx->heavy_grid;
  const int grid_heavy2 = grid_heavy > 32 ? 32 : grid_heavy;  // second heavy launch of the screened pipeline: late escalations
  if (fused && ctx->bulk_grid > 0 && grid > ctx->bulk_grid) grid = ctx->bulk_grid;
  if (getenv("CFS_DEBUG")) fprintf(stderr, "[cfs] solve: B=%d fused=%d warp=%d cfg=%d zs=%d grid=%d grid_heavy=%d\n", B, (int)fused, (int)warp, ctx->warp_cfg, a.warp_zs, grid, grid_heavy);
  // spill slabs of the working-set inverse: the warp tier has its own (zslab); the CTA tiers need n x n per CTA, and the two
  // heavy launches of the screened pipeline can overlap, so they get disjoint halves
  const int slab_ctas = fused ? ((warp ? 0 : grid) > (1 + CFS_MAX_SCREEN) * grid_heavy ? grid : (1 + CFS_MAX_SCREEN) * grid_heavy) : grid;
  if ((rc = ensure(ctx, ctx->slab, sizeof(double) * (size_t)n * n * slab_ctas))) return rc;
  a.slab = ptr<double>(ctx->slab);

  const bool detail = ctx->timing_level >= 2;
  const size_t need_ev = detail ? (size_t)3 * max_outer + 3 : 0;
  while (ctx->ev.size() < need_ev) {
    cudaEvent_t e;
    CU(cudaEventCreate(&e));
    ctx->ev.push_back(e);
  }
  int launches = 0;
  CU(cudaEventRecord(ctx->ev_a, st));
  CU(cudaMemsetAsync(cnt, 0, sizeof(int) * 64, st));
  CU(cudaMemsetAsync(ctx->qpsteps.p, 0, sizeof(long long) * 32, st));
  CU(cudaMemsetAsync(ctx->probsteps.p, 0, sizeof(int) * B, st));
  a.list_cur = ptr<int>(ctx->listA); a.count_cur = cnt + 0;
  a.list_next = ptr<int>(ctx->listB); a.count_next = cnt + 1;
  a.work_counter = cnt + 2;
  if (fused) {
    NvtxRange nvtx_solve("cfs:fused solve (screen | bulk | heavy)");
    const bool screen = warp && ctx->screen && !ctx->heavy_skip;
    const bool side = ctx->heavy_stream && ctx->heavy_prio && !detail;  // heavy tier on its own highest-priority stream
    // one persistent kernel: every CTA carries a problem through all its outer iterations (k_fused.cu)
    CU(launch_dgemm(n, B, n, -1.0, ctx->dG + (size_t)2 * n * np + 2 * n, np, false, ff, n, a.u0, n, st)); ++launches;
    CU(launch_v0(a, st)); ++launches;
    a.esc_list = ptr<int>(ctx->listA);
    a.esc_count = cnt + 5;
    a.work_counter2 = cnt + 4;
    a.esc_steps = ctx->esc_steps;
    // work order: a scheduling heuristic from the reference line only; it ignores margin_off (the offsets change no result)
    if (ctx->lpt && O > 0 && B > 1) {  // listB / flags are free in the fused path: work order + its scratch
      CU(launch_work_order(ctx->dtab, nj, O, B, H, xref, a.margin_is_D, ptr<int>(ctx->flags), ptr<int>(ctx->listB), st));
      launches += 2;
      a.order = ptr<int>(ctx->listB);
    }
    if (detail) CU(cudaEventRecord(ctx->ev[0], st));
    if (screen) {
      // Screening passes: outer iteration 1 (then 2, ... for ctx->screen > 1) of every problem in a launch of its own.  The long
      // dual chains (almost all of them infeasibility certificates of an early linearisation) reach the heavy tier a fraction
      // of a millisecond into the batch and run -- each pass's escalations on their own highest-priority stream -- concurrently
      // with the rest of the work instead of after it; everything unfinished continues in the next launch.
      //   lists in ctx->cont (B ints each): [0] cont A, [1] cont B, [2] touch flags, [3 + p] escalations of pass p
      //   counters: cnt[16 + 4 p + {0,1,2,3}] = cont count, work queue, escalation count, heavy work queue of pass p
      int *ext = ptr<int>(ctx->cont);
      const int npass = ctx->screen > CFS_MAX_SCREEN ? CFS_MAX_SCREEN : ctx->screen;
      const size_t slab_h = (size_t)n * n;
      SolveArgs ap = a;
      ap.touch = ext + 2 * (size_t)B;
      int heavy_launches = 0;
      SolveArgs heavy_args[CFS_MAX_SCREEN + 1];
      bool on_side[CFS_MAX_SCREEN + 1] = {false, false, false, false};
      for (int p = 0; p <= npass; ++p) {  // p < npass: screening pass of iteration p + 1; p == npass: the rest
        int *c4 = cnt + 16 + 4 * p;
        ap.phase = p == 0 ? 1 : 2;
        ap.it_stop = p < npass ? p + 1 : 0;
        ap.cont_list = ext + (size_t)((p + 1) & 1) * B;   // written by the previous pass
        ap.cont_count = p ? cnt + 16 + 4 * (p - 1) : nullptr;
        ap.cont_out = ext + (size_t)(p & 1) * B;
        ap.cont_out_count = c4;
        ap.work_counter = c4 + 1;
        ap.esc_list = ext + (3 + (size_t)p) * B;
        ap.esc_count = c4 + 2;
        ap.work_counter2 = c4 + 3;
        CU(launch_warp(ap, grid, ctx->warp_cfg, st)); ++launches;
        if (detail && p == npass) CU(cudaEventRecord(ctx->ev[1], st));
        heavy_args[p] = ap;  // heavy tier over this pass's escalation list; disjoint spill slabs (the launches can overlap)
        heavy_args[p].slab = a.slab + slab_h * (size_t)(p == 0 ? 0 : grid_heavy + (p - 1) * grid_heavy2);
        cudaStream_t hs = (side && p < npass) ? ctx->heavy_streams[p] : nullptr;
        if (hs) {
          CU(cudaEventRecord(ctx->ev_pass[p], st));
          CU(cudaStreamWaitEvent(hs, ctx->ev_pass[p], 0));
          CU(launch_fused(heavy_args[p], p == 0 ? grid_heavy : grid_heavy2, heavy_tier, hs)); ++launches;
          CU(cudaEventRecord(ctx->ev_hdone[p], hs));
          on_side[p] = true;
          ++heavy_launches;
        }
      }
      for (int p = 0; p <= npass; ++p)  // the last pass's escalations (and, without side streams, all of them) follow the warp tier
        if (!on_side[p]) { CU(launch_fused(heavy_args[p], p == 0 ? grid_heavy : grid_heavy2, heavy_tier, st)); ++launches; }
      for (int p = 0; p < npass; ++p)
        if (on_side[p]) CU(cudaStreamWaitEvent(st, ctx->ev_hdone[p], 0));
    } else {
      CU(warp ? launch_warp(a, grid, ctx->warp_cfg, st) : launch_fused(a, grid, 0, st)); ++launches;  // bulk tier: every problem
      if (detail) CU(cudaEventRecord(ctx->ev[1], st));
      // heavy tier: the (device-side) escalation list, usually < 1 % of the problems.  It runs on a highest-priority stream
      // so that, with several contexts in flight, its few CTAs (one per SM) are placed before another context's bulk tier
      // refills the SMs.
      if (ctx->heavy_skip) {
      } else if (side) {
        CU(cudaEventRecord(ctx->ev_bulk, st));
        CU(cudaStreamWaitEvent(ctx->heavy_stream, ctx->ev_bulk, 0));
        CU(launch_fused(a, grid_heavy, heavy_tier, ctx->heavy_stream)); ++launches;
        CU(cudaEventRecord(ctx->ev_heavy, ctx->heavy_stream));
        CU(cudaStreamWaitEvent(st, ctx->ev_heavy, 0));
      } else {
        CU(launch_fused(a, grid_heavy, heavy_tier, st)); ++launches;
      }
    }
    if (detail) CU(cudaEventRecord(ctx->ev[2], st));
    ctx->fused_last = true;
    CU(cudaEventRecord(ctx->ev_b, st));
    ctx->stats.launches = launches;
    return 0;
  }
  ctx->fused_last = false;
  // launch-per-iteration path: QP by one warp per problem where its shared-memory regions fit (k_qp_warp)
  bool qpw = false;
  int grid_w = 0;
  if (ctx->use_warp && ctx->use_warp_lockstep) {
    for (int zs = 3; zs >= 1 && !qpw; --zs) {
      a.warp_zs = zs;
      qpw = qp_warp_supported(a);
    }
    if (qpw) {
      grid_w = qp_warp_max_grid(a, ctx->device);
      if (grid_w > (B + 3) / 4) grid_w = (B + 3) / 4;
      qpw = grid_w > 0;
    }
    if (qpw) {
      if ((rc = ensure(ctx, ctx->zslab, warp_slab_bytes_per_warp(a) * (size_t)grid_w * 4))) return rc;
      a.zslab = ptr<double>(ctx->zslab);
      a.esc_list = ptr<int>(ctx->cont);
      a.esc_count = cnt + 5;
    }
  }
  CU(launch_solve_init(a, st)); ++launches;
  if (psg) {
    CU(cudaMemsetAsync(a.w, 0, sizeof(double) * (size_t)n * B, st));  // QQ*u at u = 0
  } else {
    // u0 = -QQ^{-1} FF : the control block of G is QQ^{-1}
    CU(launch_dgemm(n, B, n, -1.0, ctx->dG + (size_t)2 * n * np + 2 * n, np, false, ff, n, a.u0, n, st)); ++launches;
    CU(launch_v0(a, st)); ++launches;
  }

  GradArgs g = traj_grad_args(ctx, B, x, a.dist, a.grad, a.flags);
  for (int it = 1; it <= max_outer; ++it) {
    NvtxRange nvtx_it("cfs:outer iteration (gradient | QP)");
    a.outer_iter = it;
    g.list = a.list_cur;
    g.count = a.count_cur;
    if (detail) CU(cudaEventRecord(ctx->ev[3 * (it - 1)], st));
    if (O > 0) {
      CU(grad == CFS_GRAD_DERIVEST ? launch_grad_derivest(g, st) : launch_grad_numjac(g, st)); ++launches;
    }
    if (detail) CU(cudaEventRecord(ctx->ev[3 * (it - 1) + 1], st));
    if (psg) { CU(launch_psg_point(a, st)); ++launches; }
    if (qpw) {
      // warp-per-problem QP (k_qp_warp); the few problems whose working set outgrows it are redone by the CTA kernel
      CU(cudaMemsetAsync(cnt + 4, 0, 2 * sizeof(int), st));
      CU(launch_qp_warp(a, grid_w, st)); ++launches;
      SolveArgs ae = a;
      ae.list_cur = a.esc_list;
      ae.count_cur = a.esc_count;
      ae.work_counter = cnt + 4;
      CU(launch_qp(ae, grid < 32 ? grid : 32, st)); ++launches;
    } else {
      CU(launch_qp(a, grid, st)); ++launches;
    }
    if (psg) {  // w = QQ*u for EVAL.get_cost now and for the next PSG step
      CU(launch_dgemm(n, B, n, 1.0, ctx->dQQraw, n, false, a.u, n, a.w, n, st)); ++launches;
      CU(launch_psg_cost(a, st)); ++launches;
    }
    if (detail) CU(cudaEventRecord(ctx->ev[3 * (it - 1) + 2], st));
    // swap lists; reset the consumed counter and the work queue
    std::swap(a.list_cur, a.list_next);
    std::swap(a.count_cur, a.count_next);
    CU(cudaMemsetAsync(a.count_next, 0, sizeof(int), st));
    CU(cudaMemsetAsync(a.work_counter, 0, sizeof(int), st));
  }
  CU(launch_finalize(a, st)); ++launches;
  CU(cudaEventRecord(ctx->ev_b, st));
  ctx->stats.launches = launches;
  return 0;
}

static int collect_stats(cfs_ctx *ctx, int B, int max_outer, const int *d_iters, const int *d_status) {
  cudaStream_t st = ctx->stream;
  long long steps[2] = {0, 0};
  int cnt[64] = {0};
  std::vector<int> it(B), stt(B);
  CU(cudaMemcpyAsync(stt.data(), d_status, sizeof(int) * B, cudaMemcpyDeviceToHost, st));
  CU(cudaMemcpyAsync(steps, ctx->qpsteps.p, sizeof(steps), cudaMemcpyDeviceToHost, st));
  CU(cudaMemcpyAsync(cnt, ctx->counters.p, sizeof(cnt), cudaMemcpyDeviceToHost, st));
  CU(cudaMemcpyAsync(it.data(), d_iters, sizeof(int) * B, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  float ms = 0;
  cudaEventElapsedTime(&ms, ctx->ev_a, ctx->ev_b);
  ctx->stats.ms_total = ms;
  ctx->stats.qp_steps = steps[0];
  ctx->stats.max_active = cnt[3];
  if (getenv("CFS_DEBUG"))
    fprintf(stderr, "[cfs] batch done: escalations per launch %d %d %d %d, continued after each screening pass %d %d %d\n", cnt[18], cnt[22],
            cnt[26], cnt[30], cnt[16], cnt[20], cnt[24]);
  long long pit = 0, gev = 0;
  for (int b = 0; b < B; ++b) {
    pit += it[b];
    gev += it[b] + (((stt[b] & 0xFF) >= 2) ? 1 : 0);  // a failed QP still consumed one gradient pass
  }
  ctx->stats.problem_iters = pit;
  ctx->stats.grad_waypoints = gev * ctx->H * ctx->nobs;
  ctx->stats.ms_grad = ctx->stats.ms_qp = 0;
  ctx->stats.ms_h2d = ctx->stats.ms_d2h = 0;  // a host form's copy times follow in flush_staged
  ctx->stats.ms_bulk = ctx->stats.ms_heavy = 0;
  if (ctx->timing_level >= 2 && ctx->fused_last && ctx->ev.size() >= 3) {
    float a = 0, b = 0;
    cudaEventElapsedTime(&a, ctx->ev[0], ctx->ev[1]);
    cudaEventElapsedTime(&b, ctx->ev[1], ctx->ev[2]);
    ctx->stats.ms_bulk = a;
    ctx->stats.ms_heavy = b;
  }
  ctx->it_grad_ms.clear();
  ctx->it_qp_ms.clear();
  if (ctx->timing_level >= 2 && !ctx->fused_last && ctx->ev.size() >= (size_t)3 * max_outer) {
    for (int k = 0; k < max_outer; ++k) {
      float a = 0, b = 0;
      cudaEventElapsedTime(&a, ctx->ev[3 * k], ctx->ev[3 * k + 1]);
      cudaEventElapsedTime(&b, ctx->ev[3 * k + 1], ctx->ev[3 * k + 2]);
      ctx->stats.ms_grad += a;
      ctx->stats.ms_qp += b;
      ctx->it_grad_ms.push_back(a);
      ctx->it_qp_ms.push_back(b);
    }
  }
  return 0;
}

// Host-side copy between a caller's pageable buffer and the context's pinned staging area.  One thread moves ~10 GB/s, a
// fraction of what the PCIe link takes (the pageable e2e figure of round 1 was bound by exactly this memcpy): large copies are
// split over up to four short-lived threads.
static void host_copy(void *dst, const void *src, size_t bytes) {
  const size_t chunk_min = (size_t)2 << 20;
  unsigned hw = std::thread::hardware_concurrency();
  size_t nt = bytes / chunk_min;
  if (nt > 4) nt = 4;
  if (hw && nt > hw) nt = hw;
  if (nt < 2) {
    memcpy(dst, src, bytes);
    return;
  }
  const size_t per = ((bytes / nt) + 4095) & ~(size_t)4095;
  std::thread th[3];
  size_t started = 0;
  for (size_t k = 1; k < nt; ++k) {
    const size_t o = k * per;
    if (o >= bytes) break;
    const size_t len = (k + 1 == nt || o + per > bytes) ? bytes - o : per;
    th[started++] = std::thread([=] { memcpy(static_cast<char *>(dst) + o, static_cast<const char *>(src) + o, len); });
  }
  memcpy(dst, src, per < bytes ? per : bytes);
  for (size_t k = 0; k < started; ++k) th[k].join();
}

// ---- the solve family: cfs_solve_batch*, cfs_solve_start_goal*, cfs_solve_routes*, cfs_solve_batch_margins*, cfs_solve_checked*
// Every entry describes its call (SolveCall) and hands it to one validator (check_solve), one enqueue on device pointers
// (enqueue_solve) and, for a host form, the transfer path (upload, then Transfer::d2h).
enum SolveForm { FORM_ARRAYS, FORM_START_GOAL, FORM_ROUTES };

// The problems of a call: the reference's per-problem arrays, or start/goal pairs or routes from which the device builds them
// (main_FANUC.m:38-49,98-103; RRTstar_CFS.m:96-163).  Routes are nj x W x B with route_len[b] valid columns (NULL: all W);
// need_len: the entry requires route_len.  noise and margin_off may be NULL.
struct SolveIn {
  SolveForm form;
  const double *x0, *ff, *caug, *xref, *theta0, *thetag, *routes;
  int W;
  const int *route_len;
  bool need_len;
  const double *noise, *margin_off;
};
static SolveIn arrays_in(const double *x0, const double *ff, const double *caug, const double *xref, const double *noise,
                         const double *margin_off = nullptr) {
  return {FORM_ARRAYS, x0, ff, caug, xref, nullptr, nullptr, nullptr, 0, nullptr, false, noise, margin_off};
}
static SolveIn start_goal_in(const double *theta0, const double *thetag, const double *noise) {
  return {FORM_START_GOAL, nullptr, nullptr, nullptr, nullptr, theta0, thetag, nullptr, 0, nullptr, false, noise, nullptr};
}
static SolveIn routes_in(const double *routes, int W, const int *route_len, bool need_len, const double *noise) {
  return {FORM_ROUTES, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, routes, W, route_len, need_len, noise, nullptr};
}
struct SolveOut {  // x and e_u_hist may be NULL in a host form (not copied back)
  double *u, *x, *cost_hist, *e_u_hist;
  int *iters, *status;
};
struct CheckedIo {  // the checked solve's arguments and its outputs beyond SolveOut (margin_off may be NULL)
  double eta;
  int max_evals, rounds;
  double gain;
  int *verdict;
  double *t_hit, *cmin;
  int *rounds_used;
  double *margin_off;
};
struct SolveCall {
  const char *who;  // the public entry, named in the error messages
  bool device;      // every pointer a device pointer
  int B, solver, grad;
  double eps_outer;
  int max_outer;
  double alpha;
  SolveIn in;
  SolveOut out;
  const CheckedIo *chk = nullptr;  // the checked solve only
};

// The batch whose statistics cfs_wait collects (d: the call on device pointers; host: a host form, whose copy times are
// collected too), or none (d = NULL).  The only writer of ctx->pending.
static void set_pending(cfs_ctx *ctx, const SolveCall *d = nullptr, bool host = false) {
  ctx->pending = {};
  if (!d) return;
  ctx->pending.active = true;
  ctx->pending.host = host;
  ctx->pending.B = d->B;
  ctx->pending.max_outer = d->max_outer;
  ctx->pending.d_iters = d->out.iters;
  ctx->pending.d_status = d->out.status;
}

// After the stream has synchronised: the staged results to the caller's buffers and, for a host form, the times of its copies
static void flush_staged(cfs_ctx *ctx, bool host) {
  for (const cfs_ctx::CopyBack &cb : ctx->copy_back) host_copy(cb.dst, cb.src, cb.bytes);
  ctx->copy_back.clear();
  if (!host) return;
  float a = 0, b = 0;
  cudaEventElapsedTime(&a, ctx->ev_h[0], ctx->ev_h[1]);
  cudaEventElapsedTime(&b, ctx->ev_h[2], ctx->ev_h[3]);
  ctx->stats.ms_h2d = a;
  ctx->stats.ms_d2h = b;
}

static int finish_pending(cfs_ctx *ctx) {
  if (!ctx->pending.active) return 0;
  const auto p = ctx->pending;
  set_pending(ctx);
  int rc = collect_stats(ctx, p.B, p.max_outer, p.d_iters, p.d_status);
  flush_staged(ctx, p.host);
  return rc;
}

extern "C" int cfs_wait(cfs_ctx *ctx) {
  if (!ctx) return CFS_E_ARG;
  CU(cudaSetDevice(ctx->device));
  if (!ctx->pending.active) {
    CU(cudaStreamSynchronize(ctx->stream));
    return 0;
  }
  return finish_pending(ctx);
}

static bool is_pinned_host(const void *p) {
  if (!p) return true;
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return at.type == cudaMemoryTypeHost || at.type == cudaMemoryTypeManaged;
}

static int ensure_stage(cfs_ctx *ctx, void *&p, size_t &cap, size_t bytes) {
  if (bytes <= cap) return 0;
  if (p) cudaFreeHost(p);
  p = nullptr;
  cap = 0;
  cudaError_t e = cudaHostAlloc(&p, bytes, cudaHostAllocDefault);
  if (e != cudaSuccess) return fail(ctx, CFS_E_NOMEM, "cudaHostAlloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
  cap = bytes;
  return 0;
}

// H2D of one input: in place when the caller's buffer is pinned, else through the context's pinned staging area
struct StageIn {
  cfs_ctx *ctx;
  bool use;
  size_t off = 0;
  cudaError_t put(void *dev, const void *host, size_t bytes, cudaStream_t st) {
    if (!host || bytes == 0) return cudaSuccess;
    const void *src = host;
    if (use) {
      void *slot = static_cast<char *>(ctx->stage_in) + off;
      host_copy(slot, host, bytes);
      off += (bytes + 255) / 256 * 256;
      src = slot;
    }
    return cudaMemcpyAsync(dev, src, bytes, cudaMemcpyHostToDevice, st);
  }
};
struct StageOut {
  cfs_ctx *ctx;
  bool use;
  size_t off = 0;
  cudaError_t get(void *host, const void *dev, size_t bytes, cudaStream_t st) {
    if (!host || bytes == 0) return cudaSuccess;
    void *dst = host;
    if (use) {
      dst = static_cast<char *>(ctx->stage_out) + off;
      off += (bytes + 255) / 256 * 256;
      ctx->copy_back.push_back({host, dst, bytes});
    }
    return cudaMemcpyAsync(dst, dev, bytes, cudaMemcpyDeviceToHost, st);
  }
};

namespace {  // internal linkage: none of this is part of the library's exported symbols

// The one transfer path of every host-pointer entry: copies between caller buffers and device buffers.  With stage set (the
// solve family), pageable caller buffers go through the context's pinned staging area (one memcpy each way) so that every copy
// is truly asynchronous; pinned / registered buffers are used in place.  A NULL caller buffer is not copied.  Staged results
// reach the caller's buffers in flush_staged, after the stream has synchronised.
struct Transfer {
  struct In { const void *host; void *dev; size_t bytes; };
  struct Out { void *host; const void *dev; size_t bytes; };
  std::vector<In> in;
  std::vector<Out> out;
  StageOut sout{nullptr, false};
  // Off for the synchronous entries (Area): their call waits for its copies anyway, and the driver's own copy from pageable
  // memory overlaps its staging memcpy with the DMA, where the staging area copies first and transfers after (measured on a
  // B200: cfs_nodes_feasible, N = 100000, 0.49 ms staged against 0.43 ms direct)
  bool stage = true;

  // the staging decision of both directions, the staging area they take, and the H2D copies
  int h2d(cfs_ctx *ctx) {
    auto staged = [](const auto &copies, size_t &bytes) {  // -> some caller buffer is pageable; bytes: the staging area they take
      bool pageable = false;
      for (const auto &e : copies)
        if (e.host && e.bytes) { bytes += (e.bytes + 255) / 256 * 256; pageable = pageable || !is_pinned_host(e.host); }
      return pageable;
    };
    size_t in_bytes = 0, out_bytes = 0;
    StageIn sin{ctx, stage && staged(in, in_bytes)};
    sout = {ctx, stage && staged(out, out_bytes)};
    int rc;
    if (sin.use && (rc = ensure_stage(ctx, ctx->stage_in, ctx->stage_in_cap, in_bytes))) return rc;
    if (sout.use && (rc = ensure_stage(ctx, ctx->stage_out, ctx->stage_out_cap, out_bytes))) return rc;
    ctx->copy_back.clear();
    for (cudaEvent_t &e : ctx->ev_h)
      if (!e) CU(cudaEventCreate(&e));
    CU(cudaEventRecord(ctx->ev_h[0], ctx->stream));
    {
      NvtxRange r("cfs:h2d");
      for (const In &e : in) CU(sin.put(e.dev, e.host, e.bytes, ctx->stream));
    }
    CU(cudaEventRecord(ctx->ev_h[1], ctx->stream));
    return 0;
  }

  int d2h(cfs_ctx *ctx) {
    CU(cudaEventRecord(ctx->ev_h[2], ctx->stream));
    {
      NvtxRange r("cfs:d2h");
      for (const Out &e : out) CU(sout.get(e.host, e.dev, e.bytes, ctx->stream));
    }
    CU(cudaEventRecord(ctx->ev_h[3], ctx->stream));
    return 0;
  }
};

// The device side of a synchronous host-pointer entry: regions of one context-owned buffer (ctx->area), each 256-byte aligned.
// A region is uploaded from a caller's buffer (in), downloaded to one (out), both (inout), or neither (tmp: a device-only
// temporary).  upload() completes the batch in flight first: its staged results wait in stage_out until then, and its
// statistics in ev_a / ev_b.
class Area {
 public:
  explicit Area(cfs_ctx *ctx) : ctx_(ctx) { io_.stage = false; }
  template <class T> Area &in(T *&dev, const T *host, size_t count) { return add<T>(dev, count, host, nullptr); }
  template <class T> Area &out(T *&dev, T *host, size_t count) { return add<T>(dev, count, nullptr, host); }
  template <class T> Area &inout(T *&dev, const T *host_in, T *host_out, size_t count) { return add<T>(dev, count, host_in, host_out); }
  template <class T> Area &tmp(T *&dev, size_t count) { return add<T>(dev, count, nullptr, nullptr); }

  // the pending batch, the buffer, the region pointers and the H2D copies
  int upload() {
    cfs_ctx *ctx = ctx_;
    int rc;
    CU(cudaSetDevice(ctx->device));
    if ((rc = finish_pending(ctx)) || (rc = ensure(ctx, ctx->area, bytes_))) return rc;
    char *base = static_cast<char *>(ctx->area.p);
    for (const Region &r : regions_) {
      r.place(base + r.off);
      if (r.in) io_.in.push_back({r.in, base + r.off, r.bytes});
      if (r.out) io_.out.push_back({r.out, base + r.off, r.bytes});
    }
    return io_.h2d(ctx);
  }

  // the D2H copies, the synchronise and the staged results to the caller's buffers
  int download() {
    cfs_ctx *ctx = ctx_;
    int rc;
    if ((rc = io_.d2h(ctx))) return rc;
    CU(cudaStreamSynchronize(ctx->stream));
    flush_staged(ctx, false);
    return 0;
  }

 private:
  struct Region {
    size_t off, bytes;
    const void *in;
    void *out;
    std::function<void(char *)> place;
  };
  template <class T> Area &add(T *&dev, size_t count, const T *in, T *out) {
    const size_t bytes = sizeof(T) * count;
    regions_.push_back({bytes_, bytes, in, out, [&dev](char *p) { dev = reinterpret_cast<T *>(p); }});
    bytes_ += (bytes + 255) / 256 * 256;
    return *this;
  }
  cfs_ctx *ctx_;
  std::vector<Region> regions_;
  size_t bytes_ = 0;
  Transfer io_;
};

}  // namespace

static int check_traj_args(cfs_ctx *ctx, const char *who, int B, int H, double eta, int margin_is_D, int max_evals);

// The argument checks of every solve entry, in this order: the context; robot, obstacles, cost and, for the start/goal and
// routes forms, the cost blocks (CFS_E_STATE); the scalars and the checked solve's rules (CFS_E_ARG); B == 0 (0: nothing to
// enqueue); NULL required buffers and the margin offsets (CFS_E_ARG).  A device form checks the offsets on the device and
// synchronises once for that.
static int check_solve(cfs_ctx *ctx, const SolveCall &s) {
  if (!ctx) return CFS_E_ARG;
  const SolveIn &in = s.in;
  const SolveOut &o = s.out;
  const CheckedIo *c = s.chk;
  int rc = check_ready(ctx, true);
  if (rc) return fail(ctx, rc, "%s: %s", s.who, ctx->err.c_str());
  if (in.form != FORM_ARRAYS && !ctx->have_blocks)
    return fail(ctx, CFS_E_STATE, "%s: the cost must be set with cfs_set_cost_blocks", s.who);
  if (s.B < 0 || s.max_outer < 0) return fail(ctx, CFS_E_ARG, "%s: B=%d max_outer=%d", s.who, s.B, s.max_outer);
  if (s.solver != CFS_SOLVER_CFS && s.solver != CFS_SOLVER_PSGCFS) return fail(ctx, CFS_E_ARG, "%s: solver=%d", s.who, s.solver);
  if (s.grad != CFS_GRAD_NUMJAC && s.grad != CFS_GRAD_DERIVEST) return fail(ctx, CFS_E_ARG, "%s: grad=%d", s.who, s.grad);
  if (in.form == FORM_ROUTES && in.W < 2) return fail(ctx, CFS_E_ARG, "%s: W=%d", s.who, in.W);
  if (c) {  // the margin of the check is the solver's
    if ((rc = check_traj_args(ctx, s.who, s.B, ctx->H, c->eta, s.solver == CFS_SOLVER_PSGCFS, c->max_evals))) return rc;
    if (c->rounds < 0) return fail(ctx, CFS_E_ARG, "%s: rounds=%d", s.who, c->rounds);
    if (!(c->gain > 0.0) || !std::isfinite(c->gain))
      return fail(ctx, CFS_E_ARG, "%s: gain must be positive and finite (%g)", s.who, c->gain);
  }
  if (s.B == 0) return 0;
  const bool no_in = in.form == FORM_ARRAYS       ? !in.x0 || !in.ff || !in.caug || !in.xref
                     : in.form == FORM_START_GOAL ? !in.theta0 || !in.thetag
                                                  : !in.routes || (in.need_len && !in.route_len);
  if (no_in || !o.u || !o.cost_hist || !o.iters || !o.status || ((s.device || c) && !o.x) ||
      (c && (!c->verdict || !c->t_hit || !c->cmin || !c->rounds_used)))
    return fail(ctx, CFS_E_ARG, "%s: NULL buffer", s.who);
  if (!in.margin_off) return 0;
  if (s.device) {
    CU(cudaSetDevice(ctx->device));
    if ((rc = ensure(ctx, ctx->chk_ctr, 64))) return rc;
    int *bad = ptr<int>(ctx->chk_ctr) + 8, hbad = 0;
    CU(launch_offsets_bad((long long)ctx->nobs * ctx->H * s.B, in.margin_off, bad, ctx->stream));
    CU(cudaMemcpyAsync(&hbad, bad, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    if (hbad) return fail(ctx, CFS_E_ARG, "%s: margin_off has a negative or non-finite entry", s.who);
    return 0;
  }
  for (size_t e = 0, N = (size_t)ctx->nobs * ctx->H * s.B; e < N; ++e)
    if (!(in.margin_off[e] >= 0.0 && in.margin_off[e] < INFINITY))
      return fail(ctx, CFS_E_ARG, "%s: margin_off[%zu] = %g is negative or non-finite", s.who, e, in.margin_off[e]);
  return 0;
}

// The context's batch buffers of a call: the problem arrays (uploaded by a host form, built on the device by the start/goal and
// routes forms) with theta0 / thetag, and a host form's other inputs and its outputs.  Size 0: not needed.
static int ensure_batch(cfs_ctx *ctx, const SolveCall &s) {
  const SolveIn &in = s.in;
  const size_t B = s.B, nj = ctx->nj, n = ctx->n, K = s.max_outer > 0 ? s.max_outer : 1, OH = (size_t)ctx->nobs * ctx->H;
  const size_t D = sizeof(double), I = sizeof(int);
  const bool host = !s.device, built = in.form != FORM_ARRAYS, arrays = host || built;
  const CheckedIo *c = s.chk;
  const struct { DevBuf &b; size_t bytes; } bufs[] = {
      {ctx->x0, arrays ? D * 2 * nj * B : 0}, {ctx->ff, arrays ? D * n * B : 0}, {ctx->caug, arrays ? D * B : 0},
      {ctx->xref, arrays ? D * 2 * n * B : 0}, {ctx->th0, built ? D * nj * B : 0}, {ctx->thg, built ? D * nj * B : 0},
      {ctx->routes, host && in.routes ? D * nj * in.W * B : 0}, {ctx->rlen, host && in.route_len ? I * B : 0},
      {ctx->noise, host && in.noise ? D * n * K * B : 0}, {ctx->rep_off, host && in.margin_off ? D * OH * B : 0},
      {ctx->u, host ? D * n * B : 0}, {ctx->x, host ? D * 2 * n * B : 0}, {ctx->cost, host ? D * K * B : 0},
      {ctx->eu, host ? D * K * B : 0}, {ctx->iters, host ? I * B : 0}, {ctx->status, host ? I * B : 0},
      {ctx->chk_out, host && c ? (2 * D + 2 * I) * B + 64 : 0}, {ctx->rep_offo, host && c && c->margin_off ? D * OH * B : 0}};
  int rc;
  for (const auto &e : bufs)
    if ((rc = ensure(ctx, e.b, e.bytes))) return rc;
  return 0;
}

// One solve on device pointers: the start/goal and routes forms first build their problems into the context's batch buffers
// (routes: N1 cubicpolytraj resampling, then the mains' set-up), then the solver, then CFS_STATUS_NO_ROUTE for the routes
// shorter than 2 waypoints (a no-op without route_len).
static int enqueue_solve(cfs_ctx *ctx, const SolveCall &s) {
  const SolveIn &in = s.in;
  const SolveOut &o = s.out;
  const int nj = ctx->nj, H = ctx->H;
  cudaStream_t st = ctx->stream;
  const double *x0 = in.x0, *ff = in.ff, *caug = in.caug, *xref = in.xref;
  if (in.form != FORM_ARRAYS) {
    double *th0 = ptr<double>(ctx->th0), *thg = ptr<double>(ctx->thg), *bx0 = ptr<double>(ctx->x0), *bff = ptr<double>(ctx->ff),
           *bcaug = ptr<double>(ctx->caug), *bxref = ptr<double>(ctx->xref);
    if (in.form == FORM_ROUTES)
      CU(launch_resample_routes(s.B, in.W, H, nj, ctx->htab.dt, in.routes, in.route_len, th0, thg, bxref, st));
    CU(launch_build_problems(s.B, H, nj, ctx->htab.dt, ctx->dQblk, ctx->stage_w, ctx->term_w, th0, thg, bx0,
                             in.form == FORM_ROUTES ? nullptr : bxref, bff, bcaug, st));
    x0 = bx0, ff = bff, caug = bcaug, xref = bxref;
  }
  int rc = solve_device(ctx, s.B, s.solver, s.grad, x0, ff, caug, xref, in.noise, s.eps_outer, s.max_outer, s.alpha, o.u, o.x,
                        o.cost_hist, o.e_u_hist, o.iters, o.status, in.margin_off);
  if (rc) return rc;
  CU(launch_mark_no_route(s.B, in.route_len, o.status, o.iters, st));
  return 0;
}

// A host form on the context's batch buffers: the call on device pointers (d, dc) and the copies between those buffers and the
// caller's
struct HostIo {
  SolveCall d;
  CheckedIo dc;
  Transfer t;
};

// Host forms, before the enqueue: the batch buffers, the call on them and the H2D copies
static int upload(cfs_ctx *ctx, const SolveCall &s, HostIo &io) {
  int rc;
  CU(cudaSetDevice(ctx->device));
  if ((rc = finish_pending(ctx))) return rc;  // one batch in flight per context
  if ((rc = ensure_batch(ctx, s))) return rc;
  const size_t B = s.B, nj = ctx->nj, n = ctx->n, K = s.max_outer, K1 = K > 0 ? K : 1, OH = (size_t)ctx->nobs * ctx->H;
  const size_t D = sizeof(double), I = sizeof(int);
  auto up = [&](auto h, DevBuf &b, size_t bytes) {  // -> the device copy of input h (NULL: none)
    io.t.in.push_back({h, b.p, bytes});
    return h ? static_cast<decltype(h)>(b.p) : nullptr;
  };
  auto down = [&](auto h, void *dev, size_t bytes) {  // -> where output h is computed
    io.t.out.push_back({h, dev, bytes});
    return static_cast<decltype(h)>(dev);
  };
  const SolveIn &h = s.in;
  io.d = s;
  io.d.device = true;
  io.d.in = {h.form, up(h.x0, ctx->x0, D * 2 * nj * B), up(h.ff, ctx->ff, D * n * B), up(h.caug, ctx->caug, D * B),
             up(h.xref, ctx->xref, D * 2 * n * B), up(h.theta0, ctx->th0, D * nj * B), up(h.thetag, ctx->thg, D * nj * B),
             up(h.routes, ctx->routes, D * nj * h.W * B), h.W, up(h.route_len, ctx->rlen, I * B), h.need_len,
             up(h.noise, ctx->noise, D * n * K1 * B), up(h.margin_off, ctx->rep_off, D * OH * B)};
  io.d.out = {down(s.out.u, ctx->u.p, D * n * B), down(s.out.x, ctx->x.p, D * 2 * n * B),
              down(s.out.cost_hist, ctx->cost.p, D * K * B), down(s.out.e_u_hist, ctx->eu.p, D * K * B),
              down(s.out.iters, ctx->iters.p, I * B), down(s.out.status, ctx->status.p, I * B)};
  if (s.chk) {  // chk_out = t_hit | cmin (doubles) | verdict | rounds_used (ints)
    const CheckedIo &c = *s.chk;
    double *t = ptr<double>(ctx->chk_out);
    int *v = reinterpret_cast<int *>(t + 2 * B);
    io.dc = {c.eta, c.max_evals, c.rounds, c.gain, down(c.verdict, v, I * B), down(c.t_hit, t, D * B), down(c.cmin, t + B, D * B),
             down(c.rounds_used, v + B, I * B), c.margin_off && OH ? down(c.margin_off, ctx->rep_offo.p, D * OH * B) : nullptr};
    io.d.chk = &io.dc;
  }
  return io.t.h2d(ctx);
}

// Every entry but the checked solve's: a host form through the staging area, a device form on the caller's pointers;
// asynchronous, or followed by cfs_wait
static int solve(cfs_ctx *ctx, const SolveCall &s, bool wait) {
  int rc = check_solve(ctx, s);
  if (rc || s.B == 0) return rc;
  HostIo io;
  if (s.device) {
    CU(cudaSetDevice(ctx->device));
    set_pending(ctx);  // statistics of an un-waited earlier batch are dropped
    if ((rc = ensure_batch(ctx, s)) || (rc = enqueue_solve(ctx, s))) return rc;
  } else if ((rc = upload(ctx, s, io)) || (rc = enqueue_solve(ctx, io.d)) || (rc = io.t.d2h(ctx))) {
    return rc;
  }
  set_pending(ctx, s.device ? &s : &io.d, !s.device);
  return wait ? cfs_wait(ctx) : 0;
}

extern "C" int cfs_solve_batch(cfs_ctx *ctx, int B, int solver, int grad, const double *x0, const double *ff,
                               const double *caug, const double *xref, const double *noise, double eps_outer,
                               int max_outer, double alpha, double *u, double *x, double *cost_hist, double *e_u_hist,
                               int *iters, int *status) {
  return solve(ctx, {"cfs_solve_batch", false, B, solver, grad, eps_outer, max_outer, alpha,
                    arrays_in(x0, ff, caug, xref, noise), {u, x, cost_hist, e_u_hist, iters, status}}, true);
}

extern "C" int cfs_solve_batch_async(cfs_ctx *ctx, int B, int solver, int grad, const double *x0, const double *ff,
                                     const double *caug, const double *xref, const double *noise, double eps_outer,
                                     int max_outer, double alpha, double *u, double *x, double *cost_hist,
                                     double *e_u_hist, int *iters, int *status) {
  return solve(ctx, {"cfs_solve_batch_async", false, B, solver, grad, eps_outer, max_outer, alpha,
                    arrays_in(x0, ff, caug, xref, noise), {u, x, cost_hist, e_u_hist, iters, status}}, false);
}

extern "C" int cfs_solve_start_goal(cfs_ctx *ctx, int B, int solver, int grad, const double *theta0, const double *thetag,
                                    const double *noise, double eps_outer, int max_outer, double alpha, double *u, double *x,
                                    double *cost_hist, double *e_u_hist, int *iters, int *status) {
  return solve(ctx, {"cfs_solve_start_goal", false, B, solver, grad, eps_outer, max_outer, alpha,
                    start_goal_in(theta0, thetag, noise), {u, x, cost_hist, e_u_hist, iters, status}}, true);
}

extern "C" int cfs_solve_start_goal_async(cfs_ctx *ctx, int B, int solver, int grad, const double *theta0, const double *thetag,
                                          const double *noise, double eps_outer, int max_outer, double alpha, double *u,
                                          double *x, double *cost_hist, double *e_u_hist, int *iters, int *status) {
  return solve(ctx, {"cfs_solve_start_goal_async", false, B, solver, grad, eps_outer, max_outer, alpha,
                    start_goal_in(theta0, thetag, noise), {u, x, cost_hist, e_u_hist, iters, status}}, false);
}

extern "C" int cfs_solve_routes(cfs_ctx *ctx, int B, int W, int solver, int grad, const double *routes, const double *noise,
                                double eps_outer, int max_outer, double alpha, double *u, double *x, double *cost_hist,
                                double *e_u_hist, int *iters, int *status) {
  return solve(ctx, {"cfs_solve_routes", false, B, solver, grad, eps_outer, max_outer, alpha,
                    routes_in(routes, W, nullptr, false, noise), {u, x, cost_hist, e_u_hist, iters, status}}, true);
}

extern "C" int cfs_solve_routes_async(cfs_ctx *ctx, int B, int W, int solver, int grad, const double *routes, const double *noise,
                                      double eps_outer, int max_outer, double alpha, double *u, double *x, double *cost_hist,
                                      double *e_u_hist, int *iters, int *status) {
  return solve(ctx, {"cfs_solve_routes_async", false, B, solver, grad, eps_outer, max_outer, alpha,
                    routes_in(routes, W, nullptr, false, noise), {u, x, cost_hist, e_u_hist, iters, status}}, false);
}

extern "C" int cfs_solve_routes_var(cfs_ctx *ctx, int B, int W, const int *route_len, int solver, int grad, const double *routes,
                                    const double *noise, double eps_outer, int max_outer, double alpha, double *u, double *x,
                                    double *cost_hist, double *e_u_hist, int *iters, int *status) {
  return solve(ctx, {"cfs_solve_routes_var", false, B, solver, grad, eps_outer, max_outer, alpha,
                    routes_in(routes, W, route_len, true, noise), {u, x, cost_hist, e_u_hist, iters, status}}, true);
}

extern "C" int cfs_solve_routes_var_async(cfs_ctx *ctx, int B, int W, const int *route_len, int solver, int grad,
                                          const double *routes, const double *noise, double eps_outer, int max_outer, double alpha,
                                          double *u, double *x, double *cost_hist, double *e_u_hist, int *iters, int *status) {
  return solve(ctx, {"cfs_solve_routes_var_async", false, B, solver, grad, eps_outer, max_outer, alpha,
                    routes_in(routes, W, route_len, true, noise), {u, x, cost_hist, e_u_hist, iters, status}}, false);
}

extern "C" int cfs_solve_routes_device(cfs_ctx *ctx, int B, int W, const int *route_len, int solver, int grad, const double *routes,
                                       const double *noise, double eps_outer, int max_outer, double alpha, double *u, double *x,
                                       double *cost_hist, double *e_u_hist, int *iters, int *status, int sync) {
  return solve(ctx, {"cfs_solve_routes_device", true, B, solver, grad, eps_outer, max_outer, alpha,
                    routes_in(routes, W, route_len, false, noise), {u, x, cost_hist, e_u_hist, iters, status}}, sync);
}

extern "C" int cfs_solve_batch_device(cfs_ctx *ctx, int B, int solver, int grad, const double *x0, const double *ff,
                                      const double *caug, const double *xref, const double *noise, double eps_outer,
                                      int max_outer, double alpha, double *u, double *x, double *cost_hist,
                                      double *e_u_hist, int *iters, int *status, int sync) {
  return solve(ctx, {"cfs_solve_batch_device", true, B, solver, grad, eps_outer, max_outer, alpha,
                    arrays_in(x0, ff, caug, xref, noise), {u, x, cost_hist, e_u_hist, iters, status}}, sync);
}

extern "C" int cfs_solve_batch_margins(cfs_ctx *ctx, int B, int solver, int grad, const double *x0, const double *ff,
                                       const double *caug, const double *xref, const double *noise, const double *margin_off,
                                       double eps_outer, int max_outer, double alpha, double *u, double *x, double *cost_hist,
                                       double *e_u_hist, int *iters, int *status) {
  return solve(ctx, {"cfs_solve_batch_margins", false, B, solver, grad, eps_outer, max_outer, alpha,
                    arrays_in(x0, ff, caug, xref, noise, margin_off), {u, x, cost_hist, e_u_hist, iters, status}}, true);
}

extern "C" int cfs_solve_batch_margins_device(cfs_ctx *ctx, int B, int solver, int grad, const double *x0, const double *ff,
                                              const double *caug, const double *xref, const double *noise, const double *margin_off,
                                              double eps_outer, int max_outer, double alpha, double *u, double *x,
                                              double *cost_hist, double *e_u_hist, int *iters, int *status, int sync) {
  return solve(ctx, {"cfs_solve_batch_margins_device", true, B, solver, grad, eps_outer, max_outer, alpha,
                    arrays_in(x0, ff, caug, xref, noise, margin_off), {u, x, cost_hist, e_u_hist, iters, status}}, sync);
}

extern "C" int cfs_resample_routes(cfs_ctx *ctx, int B, int W, int H, const double *routes, double *sampled) {
  if (!ctx) return CFS_E_ARG;
  int rc = check_ready(ctx, false);
  if (rc) return rc;
  if (B < 0 || W < 2 || H < 1 || (B > 0 && (!routes || !sampled))) return fail(ctx, CFS_E_ARG, "cfs_resample_routes: bad argument");
  if (B == 0) return 0;
  const size_t nj = ctx->nj;
  cudaStream_t st = ctx->stream;
  double *d_routes, *th0, *thg, *xs;
  Area ar(ctx);
  ar.in(d_routes, routes, nj * W * B).tmp(th0, nj * B).tmp(thg, nj * B).tmp(xs, 2 * nj * H * B);
  if ((rc = ar.upload())) return rc;
  CU(launch_resample_routes(B, W, H, nj, ctx->htab.dt, d_routes, nullptr, th0, thg, xs, st));
  // the one strided output, gathered straight into the caller's buffer: sampled (nj x (H+1) x B), column 0 = theta0,
  // columns 1..H = the theta rows of x_
  CU(cudaMemcpy2DAsync(sampled, sizeof(double) * nj * (H + 1), th0, sizeof(double) * nj, sizeof(double) * nj, B,
                       cudaMemcpyDeviceToHost, st));
  for (int i = 0; i < H; ++i)
    CU(cudaMemcpy2DAsync(sampled + nj * (i + 1), sizeof(double) * nj * (H + 1), xs + 2 * nj * i, sizeof(double) * 2 * nj * H,
                         sizeof(double) * nj, B, cudaMemcpyDeviceToHost, st));
  return ar.download();
}

// ---- CHOMP_FANUC (Lib/CHOMP_FANUC.m), k_chomp.cu ----------------------------------------------------------------------
extern "C" int cfs_chomp_batch(cfs_ctx *ctx, int B, const double *x0, const double *ff, const double *caug, const double *xref,
                               const double *u_init, double alpha, int max_outer, double *u, double *x, double *cost_hist,
                               double *e_u_hist, int *iters, int *status) {
  if (!ctx) return CFS_E_ARG;
  int rc = check_ready(ctx, true);
  if (rc) return rc;
  if (B < 0 || max_outer < 0) return fail(ctx, CFS_E_ARG, "cfs_chomp_batch: bad argument");
  if (B == 0) return 0;
  if (!x0 || !ff || !caug || !xref || !u_init || !u || !cost_hist || !iters || !status)
    return fail(ctx, CFS_E_ARG, "cfs_chomp_batch: NULL buffer");
  const size_t nj = ctx->nj, n = ctx->n, K = max_outer, OH = (size_t)ctx->nobs * ctx->H;
  cudaStream_t st = ctx->stream;
  NvtxRange nvtx("cfs:chomp");
  double *d_x0, *d_ff, *d_caug, *d_u, *d_x, *d_w, *d_cost, *d_eu, *d_dist, *d_grad, *d_ld;
  int *d_flags;
  std::vector<int> fl(B);
  Area ar(ctx);
  ar.in(d_x0, x0, 2 * nj * B).in(d_ff, ff, n * B).in(d_caug, caug, B).inout(d_u, u_init, u, n * B).inout(d_x, xref, x, 2 * n * B)
      .tmp(d_w, n * B).out(d_cost, cost_hist, K * B).out(d_eu, e_u_hist, K * B).tmp(d_dist, OH * B).tmp(d_grad, OH * nj * B)
      .tmp(d_ld, OH * nj * B).out(d_flags, fl.data(), B);
  if ((rc = ar.upload())) return rc;
  CU(cudaMemsetAsync(d_flags, 0, sizeof(int) * B, st));
  GradArgs g = traj_grad_args(ctx, B, d_x, d_dist, d_grad, d_flags);
  g.linkdist = d_ld;
  g.no_off = 1;
  ChompArgs a;
  memset(&a, 0, sizeof(a));
  a.B = B; a.n = n; a.nj = nj; a.H = ctx->H; a.nobs = ctx->nobs; a.max_outer = K; a.alpha = alpha; a.tab = ctx->dtab;
  a.x0 = d_x0; a.ff = d_ff; a.caug = d_caug; a.u = d_u; a.x = d_x; a.w = d_w;
  a.dist = d_dist; a.grad = d_grad; a.linkdist = d_ld;
  a.cost_hist = d_cost; a.e_u_hist = d_eu;
  int launches = 0;
  CU(cudaEventRecord(ctx->ev_a, st));
  if (ctx->nobs > 0) { CU(launch_grad_derivest(g, st)); ++launches; }
  CU(launch_dgemm(n, B, n, 1.0, ctx->dQQraw, n, false, d_u, n, d_w, n, st)); ++launches;
  for (int it = 1; it <= max_outer; ++it) {
    a.it = it;
    CU(launch_chomp_step(a, st)); ++launches;
    if (ctx->nobs > 0) { CU(launch_grad_derivest(g, st)); ++launches; }
    CU(launch_dgemm(n, B, n, 1.0, ctx->dQQraw, n, false, d_u, n, d_w, n, st)); ++launches;
    CU(launch_chomp_cost(a, st)); ++launches;
  }
  CU(cudaEventRecord(ctx->ev_b, st));
  if ((rc = ar.download())) return rc;
  for (int b = 0; b < B; ++b) {
    iters[b] = max_outer;
    status[b] = CFS_STATUS_MAX_ITER | (fl[b] & 0x100);  // stop_outer only ends at iter_O > MAX_O_ITER (CHOMP_FANUC.m:56)
  }
  float ms = 0;
  cudaEventElapsedTime(&ms, ctx->ev_a, ctx->ev_b);
  ctx->stats.ms_total = ms;
  ctx->stats.launches = launches;
  return 0;
}

// Development aid (dev/timeline.py; not part of include/cfs_b200.h): where the stages of the last fused solve of `ctx` fell on the
// device's time axis, in ms after the START of the last solve of `ref` (another context of the same device):
// out = {solve enqueued work starts, screening launch done, heavy launch #1 done, everything done}.  Call after cfs_wait.
extern "C" int cfs_dev_timeline(cfs_ctx *ctx, cfs_ctx *ref, double *out4) {
  if (!ctx || !ref || !out4) return CFS_E_ARG;
  cudaEvent_t ev[4] = {ctx->ev_a, ctx->ev_pass[0], ctx->ev_hdone[0], ctx->ev_b};
  for (int k = 0; k < 4; ++k) {
    float ms = 0;
    out4[k] = (ev[k] && cudaEventElapsedTime(&ms, ref->ev_a, ev[k]) == cudaSuccess) ? ms : -1.0;
  }
  cudaGetLastError();
  return 0;
}

// ---- direct kernels -------------------------------------------------------------------------------------------------
// cfs_dist_grad and cfs_time_dist_grad: theta uploaded, and the distance/gradient kernel with one "problem" per configuration so
// that flags are per configuration: dist (n_obs x N) is dist[j + O * prob].  NULL outputs are computed and not copied back.
static int config_grad(cfs_ctx *ctx, Area &ar, int N, const double *theta, double *dist, int *linkid, double *grad, int *flags,
                       GradArgs &g) {
  const size_t nj = ctx->nj, O = ctx->nobs;
  double *d_theta, *d_dist, *d_grad;
  int *d_lid, *d_flags;
  ar.in(d_theta, theta, nj * N).out(d_dist, dist, O * N).out(d_grad, grad, O * N * nj).out(d_lid, linkid, O * N).out(d_flags, flags, N);
  int rc = ar.upload();
  if (rc) return rc;
  CU(cudaMemsetAsync(d_flags, 0, sizeof(int) * N, ctx->stream));
  memset(&g, 0, sizeof(g));
  g.tab = ctx->dtab; g.dv = ctx->ddv;
  g.x = d_theta;
  g.ld_prob = nj; g.ld_i = 0; g.nslots = N; g.H = 1; g.nj = nj; g.nobs = O;
  g.o_prob = O; g.o_obs = 1; g.o_i = 0;
  g.dist = d_dist; g.linkid = d_lid; g.grad = d_grad; g.flags = d_flags;
  return 0;
}

extern "C" int cfs_dist_grad(cfs_ctx *ctx, int N, int grad_mode, const double *theta, double *dist, int *linkid,
                             double *grad, int *flags) {
  if (!ctx) return CFS_E_ARG;
  int rc = check_ready(ctx, false);
  if (rc) return rc;
  if (N < 0 || (N > 0 && (!theta || !dist || !grad))) return fail(ctx, CFS_E_ARG, "cfs_dist_grad: bad argument");
  if (N == 0 || ctx->nobs == 0) return 0;
  Area ar(ctx);
  GradArgs g;
  if ((rc = config_grad(ctx, ar, N, theta, dist, linkid, grad, flags, g))) return rc;
  CU(grad_mode == CFS_GRAD_DERIVEST ? launch_grad_derivest(g, ctx->stream) : launch_grad_numjac(g, ctx->stream));
  return ar.download();
}

extern "C" int cfs_time_dist_grad(cfs_ctx *ctx, int N, int grad_mode, const double *theta, int reps, double *ms_per_launch) {
  if (!ctx || !theta || !ms_per_launch || N <= 0 || reps <= 0) return CFS_E_ARG;
  int rc = check_ready(ctx, false);
  if (rc) return rc;
  if (ctx->nobs == 0) return fail(ctx, CFS_E_STATE, "cfs_time_dist_grad: no obstacles");
  cudaStream_t st = ctx->stream;
  Area ar(ctx);
  GradArgs g;
  if ((rc = config_grad(ctx, ar, N, theta, nullptr, nullptr, nullptr, nullptr, g))) return rc;
  for (int w = 0; w < 2; ++w) CU(grad_mode == CFS_GRAD_DERIVEST ? launch_grad_derivest(g, st) : launch_grad_numjac(g, st));
  CU(cudaEventRecord(ctx->ev_a, st));
  for (int r = 0; r < reps; ++r) CU(grad_mode == CFS_GRAD_DERIVEST ? launch_grad_derivest(g, st) : launch_grad_numjac(g, st));
  CU(cudaEventRecord(ctx->ev_b, st));
  if ((rc = ar.download())) return rc;
  float ms = 0;
  cudaEventElapsedTime(&ms, ctx->ev_a, ctx->ev_b);
  *ms_per_launch = ms / reps;
  return 0;
}

// The reference's rows of CFS_FANUC.get_con for one problem, computed on the device: A (m x n, column-major) and b (m)
static int con_rows(cfs_ctx *ctx, int grad_mode, int margin_is_D, const double *x0, const double *xcur, const double *u, int m,
                    double *A, double *b) {
  const size_t nj = ctx->nj, n = ctx->n, OH = (size_t)ctx->nobs * ctx->H;
  cudaStream_t st = ctx->stream;
  double *d_x0, *d_x, *d_u, *d_dist, *d_grad, *d_A, *d_b;
  int *d_flags;
  Area ar(ctx);
  ar.in(d_x0, x0, 2 * nj).in(d_x, xcur, 2 * n).in(d_u, u, n).tmp(d_dist, OH).tmp(d_grad, OH * nj).out(d_A, A, m * n)
      .out(d_b, b, m).tmp(d_flags, 1);
  int rc = ar.upload();
  if (rc) return rc;
  CU(cudaMemsetAsync(d_flags, 0, sizeof(int), st));
  const GradArgs g = traj_grad_args(ctx, 1, d_x, d_dist, d_grad, d_flags);
  CU(grad_mode == CFS_GRAD_DERIVEST ? launch_grad_derivest(g, st) : launch_grad_numjac(g, st));
  CU(launch_get_con_rows(ctx->dtab, ctx->H, nj, ctx->nobs, ctx->has_lim, margin_is_D, d_x0, d_u, ctx->dlim, d_dist, d_grad, d_A,
                         d_b, m, st));
  return ar.download();
}

extern "C" int cfs_get_con(cfs_ctx *ctx, int grad_mode, int margin_is_D, const double *x0, const double *xcur,
                           const double *u, double *Ainq, double *binq) {
  if (!ctx) return CFS_E_ARG;
  int rc = check_ready(ctx, true);
  if (rc) return rc;
  if (!x0 || !xcur || !u || !Ainq || !binq) return fail(ctx, CFS_E_ARG, "cfs_get_con: NULL argument");
  const int nj = ctx->nj, n = ctx->n;
  const int m = ctx->nobs * ctx->H * (ctx->has_lim ? 1 + 2 * nj : 1);
  if (!ctx->has_qlim) return m > 0 ? con_rows(ctx, grad_mode, margin_is_D, x0, xcur, u, m, Ainq, binq) : 0;
  // joint position rows after the reference's rows: theta_(i+1),k <= qmax_k, then -theta_(i+1),k <= -qmin_k
  const int mt = m + 2 * n;
  std::vector<double> A0((size_t)m * n), b0(m);
  if (m > 0 && (rc = con_rows(ctx, grad_mode, margin_is_D, x0, xcur, u, m, A0.data(), b0.data()))) return rc;
  const double dt = ctx->htab.dt;
  for (int c = 0; c < n; ++c) {
    for (int r = 0; r < m; ++r) Ainq[r + (size_t)mt * c] = A0[r + (size_t)m * c];
    const int jj = c / nj, kc = c - jj * nj;
    for (int e = 0; e < n; ++e) {
      const int i = e / nj, k = e - i * nj;
      const double v = (k == kc && jj <= i) ? (0.5 * dt * dt + ((i - jj) * dt) * dt) : 0.0;
      Ainq[m + e + (size_t)mt * c] = v;
      Ainq[m + n + e + (size_t)mt * c] = -v;
    }
  }
  for (int r = 0; r < m; ++r) binq[r] = b0[r];
  for (int e = 0; e < n; ++e) {
    const int i = e / nj, k = e - i * nj;
    const double fm = x0[k] + ((i + 1) * dt) * x0[nj + k];
    binq[m + e] = ctx->hqlim[k] - fm;
    binq[m + n + e] = fm - ctx->hqlim[nj + k];
  }
  return 0;
}

extern "C" int cfs_nodes_feasible(cfs_ctx *ctx, int N, const double *theta, unsigned char *feasible, double *dmin) {
  if (!ctx) return CFS_E_ARG;
  int rc = check_ready(ctx, false);
  if (rc) return rc;
  if (N < 0 || (N > 0 && (!theta || !feasible))) return fail(ctx, CFS_E_ARG, "cfs_nodes_feasible: bad argument");
  if (N == 0) return 0;
  const size_t nj = ctx->nj;
  double *d_theta, *d_dmin;
  unsigned char *d_feas;
  Area ar(ctx);
  ar.in(d_theta, theta, nj * N).out(d_feas, feasible, N).out(d_dmin, dmin, N);
  if ((rc = ar.upload())) return rc;
  CU(launch_nodes_feasible(ctx->dtab, nj, ctx->nobs, N, d_theta, d_feas, d_dmin, ctx->stream));
  return ar.download();
}

// ---- continuous collision checks (k_check.cu) ------------------------------------------------------------------------
static_assert(CHK_CLEAR == CFS_CHECK_CLEAR && CHK_HIT == CFS_CHECK_HIT && CHK_UNDECIDED == CFS_CHECK_UNDECIDED, "verdict codes");

static int check_check_args(cfs_ctx *ctx, const char *who, int N, double eta, int margin_is_D, int max_evals) {
  if (!ctx) return CFS_E_ARG;
  int rc = check_ready(ctx, false);
  if (rc) return rc;
  if (N < 0) return fail(ctx, CFS_E_ARG, "%s: negative count %d", who, N);
  if (!(eta > 0.0) || !std::isfinite(eta)) return fail(ctx, CFS_E_ARG, "%s: eta must be positive and finite (%g)", who, eta);
  if (max_evals < 1) return fail(ctx, CFS_E_ARG, "%s: max_evals=%d", who, max_evals);
  for (int j = 0; j < ctx->nobs; ++j) {
    const double m = margin_is_D ? ctx->htab.obs[j].D : ctx->htab.obs[j].eps;
    if (!(m - eta >= 1e-4))  // below it the touch rule (|d| < 1e-4) could fire inside the certified band
      return fail(ctx, CFS_E_ARG, "%s: margin %g of obstacle %d minus eta %g is below 1e-4", who, m, j, eta);
  }
  return 0;
}

static CheckArgs check_base(cfs_ctx *ctx, int mode, int N, double eta, int margin_is_D, int max_evals) {
  CheckArgs a;
  memset(&a, 0, sizeof(a));
  a.tab = ctx->dtab; a.mode = mode; a.N = N; a.nj = ctx->nj; a.nobs = ctx->nobs;
  a.margin_is_D = margin_is_D ? 1 : 0; a.max_evals = max_evals; a.eta = eta;
  for (int k = 0; k < CFS_MAXL; ++k) a.R[k] = ctx->motion_R[k];
  a.counter = ptr<int>(ctx->chk_ctr);
  return a;
}

static int check_edges_dev(cfs_ctx *ctx, int N, const double *theta_a, const double *theta_b, double eta, int margin_is_D,
                           int max_evals, int *verdict, double *s_hit, double *cmin, int *evals) {
  int rc;
  if ((rc = ensure(ctx, ctx->chk_ctr, 64))) return rc;
  CheckArgs a = check_base(ctx, 0, N, eta, margin_is_D, max_evals);
  a.theta_a = theta_a; a.theta_b = theta_b;
  a.verdict = verdict; a.s_hit = s_hit; a.cmin = cmin; a.evals = evals;
  CU(launch_check(a, ctx->device, ctx->stream));
  return 0;
}

static int check_traj_dev(cfs_ctx *ctx, int B, int H, const double *x0, const double *x, const double *u, double eta,
                          int margin_is_D, int max_evals, int *verdict, double *t_hit, double *cmin, int *evals) {
  int rc;
  const size_t S = (size_t)B * H;
  if ((rc = ensure(ctx, ctx->chk_ctr, 64))) return rc;
  if ((rc = ensure(ctx, ctx->chk_seg, (2 * sizeof(double) + 2 * sizeof(int)) * S + 64))) return rc;
  double *ss = ptr<double>(ctx->chk_seg), *sc = ss + S;
  int *sv = reinterpret_cast<int *>(sc + S), *se = sv + S;
  CheckArgs a = check_base(ctx, 1, (int)S, eta, margin_is_D, max_evals);
  a.H = H; a.x0 = x0; a.x = x; a.u = u;
  a.verdict = sv; a.s_hit = ss; a.cmin = sc; a.evals = se;
  CU(launch_check(a, ctx->device, ctx->stream));
  CU(launch_check_reduce(B, H, ctx->htab.dt, sv, ss, sc, se, verdict, t_hit, cmin, evals, ctx->stream));
  return 0;
}

// The argument checks of cfs_check_edges and its device form: check_check_args, then (N > 0) the required buffers
static int check_edges_call(cfs_ctx *ctx, const char *who, int N, const void *theta_a, const void *theta_b, double eta,
                            int margin_is_D, int max_evals, const void *verdict, const void *s_hit, const void *cmin) {
  int rc = check_check_args(ctx, who, N, eta, margin_is_D, max_evals);
  if (rc || N == 0) return rc;
  if (!theta_a || !theta_b || !verdict || !s_hit || !cmin) return fail(ctx, CFS_E_ARG, "%s: NULL buffer", who);
  return 0;
}

extern "C" int cfs_check_edges_device(cfs_ctx *ctx, int N, const double *theta_a, const double *theta_b, double eta,
                                      int margin_is_D, int max_evals, int *verdict, double *s_hit, double *cmin, int *evals,
                                      int sync) {
  int rc = check_edges_call(ctx, "cfs_check_edges_device", N, theta_a, theta_b, eta, margin_is_D, max_evals, verdict, s_hit, cmin);
  if (rc || N == 0) return rc;
  CU(cudaSetDevice(ctx->device));
  if ((rc = check_edges_dev(ctx, N, theta_a, theta_b, eta, margin_is_D, max_evals, verdict, s_hit, cmin, evals))) return rc;
  if (sync) CU(cudaStreamSynchronize(ctx->stream));
  return 0;
}

extern "C" int cfs_check_edges(cfs_ctx *ctx, int N, const double *theta_a, const double *theta_b, double eta, int margin_is_D,
                               int max_evals, int *verdict, double *s_hit, double *cmin, int *evals) {
  int rc = check_edges_call(ctx, "cfs_check_edges", N, theta_a, theta_b, eta, margin_is_D, max_evals, verdict, s_hit, cmin);
  if (rc || N == 0) return rc;
  const size_t nj = ctx->nj;
  double *d_a, *d_b, *d_s, *d_c;
  int *d_v, *d_e;
  Area ar(ctx);
  ar.in(d_a, theta_a, nj * N).in(d_b, theta_b, nj * N).out(d_v, verdict, N).out(d_s, s_hit, N).out(d_c, cmin, N).out(d_e, evals, N);
  if ((rc = ar.upload()) || (rc = check_edges_dev(ctx, N, d_a, d_b, eta, margin_is_D, max_evals, d_v, d_s, d_c, d_e))) return rc;
  return ar.download();
}

static int check_traj_args(cfs_ctx *ctx, const char *who, int B, int H, double eta, int margin_is_D, int max_evals) {
  int rc = check_check_args(ctx, who, B, eta, margin_is_D, max_evals);
  if (rc) return rc;
  if (H < 1) return fail(ctx, CFS_E_ARG, "%s: H=%d", who, H);
  if ((long long)B * H > 0x7fffffffLL) return fail(ctx, CFS_E_ARG, "%s: B*H=%lld segments", who, (long long)B * H);
  return 0;
}

// The argument checks of cfs_check_trajectories and its device form: check_traj_args, then (B > 0) the required buffers
static int check_traj_call(cfs_ctx *ctx, const char *who, int B, int H, const void *x0, const void *x, const void *u, double eta,
                           int margin_is_D, int max_evals, const void *verdict, const void *t_hit, const void *cmin) {
  int rc = check_traj_args(ctx, who, B, H, eta, margin_is_D, max_evals);
  if (rc || B == 0) return rc;
  if (!x0 || !x || !u || !verdict || !t_hit || !cmin) return fail(ctx, CFS_E_ARG, "%s: NULL buffer", who);
  return 0;
}

extern "C" int cfs_check_trajectories_device(cfs_ctx *ctx, int B, int H, const double *x0, const double *x, const double *u,
                                             double eta, int margin_is_D, int max_evals, int *verdict, double *t_hit,
                                             double *cmin, int *evals, int sync) {
  int rc = check_traj_call(ctx, "cfs_check_trajectories_device", B, H, x0, x, u, eta, margin_is_D, max_evals, verdict, t_hit, cmin);
  if (rc || B == 0) return rc;
  CU(cudaSetDevice(ctx->device));
  if ((rc = check_traj_dev(ctx, B, H, x0, x, u, eta, margin_is_D, max_evals, verdict, t_hit, cmin, evals))) return rc;
  if (sync) CU(cudaStreamSynchronize(ctx->stream));
  return 0;
}

extern "C" int cfs_check_trajectories(cfs_ctx *ctx, int B, int H, const double *x0, const double *x, const double *u, double eta,
                                      int margin_is_D, int max_evals, int *verdict, double *t_hit, double *cmin, int *evals) {
  int rc = check_traj_call(ctx, "cfs_check_trajectories", B, H, x0, x, u, eta, margin_is_D, max_evals, verdict, t_hit, cmin);
  if (rc || B == 0) return rc;
  const size_t nj = ctx->nj, S = (size_t)B * H;
  double *d_x0, *d_x, *d_u, *d_t, *d_c;
  int *d_v, *d_e;
  Area ar(ctx);
  ar.in(d_x0, x0, 2 * nj * B).in(d_x, x, 2 * nj * S).in(d_u, u, nj * S).out(d_v, verdict, B).out(d_t, t_hit, B).out(d_c, cmin, B)
      .out(d_e, evals, B);
  if ((rc = ar.upload()) || (rc = check_traj_dev(ctx, B, H, d_x0, d_x, d_u, eta, margin_is_D, max_evals, d_v, d_t, d_c, d_e)))
    return rc;
  return ar.download();
}

// ---- the checked solve (include/cfs_b200.h) ------------------------------------------------------------------------
// The round loop.  Problem-indexed state lives in the caller's (device) buffers; the sub-batch of a round (at most B problems) in
// context buffers: rep_in = x0 | ff | caug | xref | noise | offsets, rep_out = u | x | cost | e_u | verdict | t_hit | cmin (doubles)
// then iters | status | verdict (ints), rep_list = sel | list A | list B | count.  rep_off holds the accumulated offsets of every
// problem; margin_off_out (NULL: not returned) receives the offsets of the round each returned solution comes from.
static int solve_checked_dev(cfs_ctx *ctx, const SolveCall &s) {
  const CheckedIo &c = *s.chk;
  const int B = s.B, solver = s.solver, grad = s.grad, max_outer = s.max_outer, max_evals = c.max_evals, rounds = c.rounds;
  const double eps_outer = s.eps_outer, alpha = s.alpha, eta = c.eta, gain = c.gain;
  const double *x0 = s.in.x0, *ff = s.in.ff, *caug = s.in.caug, *xref = s.in.xref, *noise = s.in.noise;
  double *u = s.out.u, *x = s.out.x, *cost_hist = s.out.cost_hist, *e_u_hist = s.out.e_u_hist, *t_hit = c.t_hit, *cmin = c.cmin,
         *margin_off_out = c.margin_off;
  int *iters = s.out.iters, *status = s.out.status, *verdict = c.verdict, *rounds_used = c.rounds_used;
  const int nj = ctx->nj, n = ctx->n, H = ctx->H, O = ctx->nobs, K = max_outer;
  const size_t OH = (size_t)O * H, nx0 = 2 * nj, N = 2 * (size_t)n, nnz = noise ? (size_t)n * K : 0;
  const int margin_is_D = solver == CFS_SOLVER_PSGCFS;
  cudaStream_t st = ctx->stream;
  int rc;
  set_pending(ctx);
  // round 0: the plain solve and its check
  if ((rc = enqueue_solve(ctx, s))) return rc;
  if ((rc = collect_stats(ctx, B, max_outer, iters, status))) return rc;  // cfs_get_stats: round 0's solve
  if ((rc = check_traj_dev(ctx, B, H, x0, x, u, eta, margin_is_D, max_evals, verdict, t_hit, cmin, nullptr))) return rc;
  CU(cudaMemsetAsync(rounds_used, 0, sizeof(int) * B, st));
  if ((rc = ensure(ctx, ctx->rep_off, sizeof(double) * (OH ? OH : 1) * B))) return rc;
  double *off = ptr<double>(ctx->rep_off);
  if (OH) CU(cudaMemsetAsync(off, 0, sizeof(double) * OH * B, st));
  if (OH && margin_off_out) CU(cudaMemsetAsync(margin_off_out, 0, sizeof(double) * OH * B, st));
  if (rounds == 0 || O == 0) return 0;

  const size_t in_row = nx0 + n + 1 + N + nnz + OH, out_row = n + N + 2 * (size_t)(K > 0 ? K : 1) + 2;
  if ((rc = ensure(ctx, ctx->rep_in, sizeof(double) * in_row * B))) return rc;
  if ((rc = ensure(ctx, ctx->rep_out, sizeof(double) * out_row * B + sizeof(int) * 3 * (size_t)B))) return rc;
  if ((rc = ensure(ctx, ctx->rep_list, sizeof(int) * (3 * (size_t)B + 2)))) return rc;
  double *sx0 = ptr<double>(ctx->rep_in), *sff = sx0 + nx0 * B, *scaug = sff + (size_t)n * B, *sxref = scaug + B,
         *snoise = sxref + N * B, *soff = snoise + nnz * B;
  const int Kc = K > 0 ? K : 1;
  double *su = ptr<double>(ctx->rep_out), *sx = su + (size_t)n * B, *sch = sx + N * B, *seu = sch + (size_t)Kc * B,
         *sth = seu + (size_t)Kc * B, *scm = sth + B;
  int *sit = reinterpret_cast<int *>(scm + B), *sst = sit + B, *sv = sst + B;
  int *sel = ptr<int>(ctx->rep_list), *lst[2] = {sel + B, sel + 2 * (size_t)B}, *d_count = sel + 3 * (size_t)B;
  CheckArgs ca = check_base(ctx, 1, B * H, eta, margin_is_D, max_evals);
  ca.H = H;
  // per-segment results of the last check of nb trajectories, as check_traj_dev lays them out in chk_seg
  auto seg_results = [&](int nb) {
    const size_t S = (size_t)nb * H;
    ca.s_hit = ptr<double>(ctx->chk_seg);
    ca.verdict = reinterpret_cast<int *>(ca.s_hit + 2 * S);
  };

  // after round 0: HIT and status < 2 -> list; increments from the round-0 check
  CU(launch_repair_select(B, verdict, status, nullptr, sel, lst[0], d_count, st));
  ca.x0 = x0; ca.x = x; ca.u = u;
  seg_results(B);
  CU(launch_repair_margins(ca, B, d_count, sel, nullptr, gain, off, st));
  int cur = 0;
  for (int r = 1; r <= rounds; ++r) {
    int c = 0;  // one count readback per round
    CU(cudaMemcpyAsync(&c, d_count, sizeof(int), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    if (c == 0) break;
    const int *L = lst[cur];
    // gather the sub-batch from the caller's original inputs (re-solved from xref, not warm-started) and the offsets
    CU(launch_rows_copy(c, L, x0, sx0, nx0, 0, nullptr, st));
    CU(launch_rows_copy(c, L, ff, sff, n, 0, nullptr, st));
    CU(launch_rows_copy(c, L, caug, scaug, 1, 0, nullptr, st));
    CU(launch_rows_copy(c, L, xref, sxref, N, 0, nullptr, st));
    if (noise) CU(launch_rows_copy(c, L, noise, snoise, nnz, 0, nullptr, st));
    CU(launch_rows_copy(c, L, off, soff, OH, 0, nullptr, st));
    if ((rc = solve_device(ctx, c, solver, grad, sx0, sff, scaug, sxref, noise ? snoise : nullptr, eps_outer, max_outer, alpha, su,
                           sx, sch, e_u_hist ? seu : nullptr, sit, sst, soff)))
      return rc;
    if ((rc = check_traj_dev(ctx, c, H, sx0, sx, su, eta, margin_is_D, max_evals, sv, sth, scm, nullptr))) return rc;
    // accepted candidates (status < 2) replace the solution; failed ones leave it and stop repairing
    CU(launch_rows_copy(c, L, su, u, n, 1, sst, st));
    CU(launch_rows_copy(c, L, sx, x, N, 1, sst, st));
    if (K > 0) {
      CU(launch_rows_copy(c, L, sch, cost_hist, K, 1, sst, st));
      if (e_u_hist) CU(launch_rows_copy(c, L, seu, e_u_hist, K, 1, sst, st));
    }
    CU(launch_ints_copy(c, L, sit, iters, 1, sst, -1, st));
    CU(launch_ints_copy(c, L, sst, status, 1, sst, -1, st));
    CU(launch_ints_copy(c, L, sv, verdict, 1, sst, -1, st));
    CU(launch_rows_copy(c, L, sth, t_hit, 1, 1, sst, st));
    CU(launch_rows_copy(c, L, scm, cmin, 1, 1, sst, st));
    CU(launch_ints_copy(c, L, nullptr, rounds_used, 1, sst, r, st));
    if (margin_off_out) CU(launch_rows_copy(c, L, soff, margin_off_out, OH, 1, sst, st));
    if (r == rounds) break;
    CU(launch_repair_select(c, sv, sst, L, sel, lst[cur ^ 1], d_count, st));
    ca.x0 = sx0; ca.x = sx; ca.u = su;
    seg_results(c);
    CU(launch_repair_margins(ca, c, d_count, sel, L, gain, off, st));
    cur ^= 1;
  }
  return 0;
}

extern "C" int cfs_solve_checked_device(cfs_ctx *ctx, int B, int solver, int grad, const double *x0, const double *ff,
                                        const double *caug, const double *xref, const double *noise, double eps_outer,
                                        int max_outer, double alpha, double eta, int max_evals, int rounds, double gain, double *u,
                                        double *x, double *cost_hist, double *e_u_hist, int *iters, int *status, int *verdict,
                                        double *t_hit, double *cmin, int *rounds_used, double *margin_off, int sync) {
  const CheckedIo c{eta, max_evals, rounds, gain, verdict, t_hit, cmin, rounds_used, margin_off};
  const SolveCall s{"cfs_solve_checked_device", true, B, solver, grad, eps_outer, max_outer, alpha,
                    arrays_in(x0, ff, caug, xref, noise), {u, x, cost_hist, e_u_hist, iters, status}, &c};
  int rc = check_solve(ctx, s);
  if (rc || B == 0) return rc;
  CU(cudaSetDevice(ctx->device));
  if ((rc = solve_checked_dev(ctx, s))) return rc;
  if (sync) CU(cudaStreamSynchronize(ctx->stream));
  return 0;
}

extern "C" int cfs_solve_checked(cfs_ctx *ctx, int B, int solver, int grad, const double *x0, const double *ff, const double *caug,
                                 const double *xref, const double *noise, double eps_outer, int max_outer, double alpha, double eta,
                                 int max_evals, int rounds, double gain, double *u, double *x, double *cost_hist, double *e_u_hist,
                                 int *iters, int *status, int *verdict, double *t_hit, double *cmin, int *rounds_used,
                                 double *margin_off) {
  const CheckedIo c{eta, max_evals, rounds, gain, verdict, t_hit, cmin, rounds_used, margin_off};
  const SolveCall s{"cfs_solve_checked", false, B, solver, grad, eps_outer, max_outer, alpha,
                    arrays_in(x0, ff, caug, xref, noise), {u, x, cost_hist, e_u_hist, iters, status}, &c};
  int rc = check_solve(ctx, s);
  if (rc || B == 0) return rc;
  HostIo io;
  if ((rc = upload(ctx, s, io)) || (rc = solve_checked_dev(ctx, io.d)) || (rc = io.t.d2h(ctx))) return rc;
  CU(cudaStreamSynchronize(ctx->stream));
  flush_staged(ctx, true);
  return 0;
}

extern "C" int cfs_nearest_steer(cfs_ctx *ctx, int n_nodes, const double *nodes, int S, const double *samples,
                                 const double *ratial, double step, int *parent, double *newnode) {
  if (!ctx) return CFS_E_ARG;
  if (!ctx->have_robot) return fail(ctx, CFS_E_STATE, "robot not set (cfs_set_robot)");
  if (n_nodes < 1 || S < 0 || !nodes || (S > 0 && (!samples || !ratial || !parent || !newnode)))
    return fail(ctx, CFS_E_ARG, "cfs_nearest_steer: bad argument");
  if (S == 0) return 0;
  const size_t nj = ctx->nj;
  double *d_nodes, *d_s, *d_r, *d_new;
  int *d_par;
  Area ar(ctx);
  ar.in(d_nodes, nodes, nj * n_nodes).in(d_s, samples, nj * S).in(d_r, ratial, nj).out(d_par, parent, S).out(d_new, newnode, nj * S);
  int rc = ar.upload();
  if (rc) return rc;
  CU(launch_nearest_steer(nj, n_nodes, d_nodes, S, d_s, d_r, step, d_par, d_new, ctx->stream));
  return ar.download();
}

// The argument checks of cfs_rrt_find_routes and its device form (have_params: the four parameter vectors, or params, given)
static int check_rrt_call(cfs_ctx *ctx, const char *who, int S, int max_iter, int nrnd, const void *x0, const void *goal,
                          const void *goal_th, bool have_params, const void *rnd, const void *routes, const void *route_len,
                          const void *n_nodes, const void *fail_out, const void *rnd_used) {
  if (!ctx) return CFS_E_ARG;
  int rc = check_ready(ctx, false);
  if (rc) return rc;
  if (S < 0 || max_iter < 1 || nrnd < 1 ||
      (S > 0 && (!x0 || !goal || !goal_th || !have_params || !rnd || !routes || !route_len || !n_nodes || !fail_out || !rnd_used)))
    return fail(ctx, CFS_E_ARG, "%s: bad argument", who);
  return 0;
}

// Both forms of cfs_rrt_find_routes on device pointers: params = region_g | region_s | sample_off | ratial (nj each); the tree
// outputs may be NULL
static int rrt_dev(cfs_ctx *ctx, int S, int star, const double *x0, const double *goal, const double *goal_th, const double *params,
                   double bi, int max_iter, const double *rnd, int nrnd, double *routes, int *route_len, int *n_nodes, int *fail_out,
                   int *rnd_used, double *tree_nodes, int *tree_parent, double *tree_total) {
  const int nj = ctx->nj;
  RrtArgs a;
  memset(&a, 0, sizeof(a));
  a.tab = ctx->dtab; a.nj = nj; a.nobs = ctx->nobs; a.star = star; a.max_iter = max_iter; a.nrnd = nrnd; a.bi = bi;
  a.x0 = x0; a.goal = goal; a.goal_th = goal_th;
  a.region_g = params; a.region_s = params + nj; a.sample_off = params + 2 * nj; a.ratial = params + 3 * nj;
  a.rnd = rnd; a.routes = routes; a.route_len = route_len; a.n_nodes = n_nodes; a.fail = fail_out; a.rnd_used = rnd_used;
  a.tree_nodes = tree_nodes; a.tree_total = tree_total; a.tree_parent = tree_parent;
  CU(launch_rrt_find_routes(a, S, ctx->stream));
  return 0;
}

extern "C" int cfs_rrt_find_routes(cfs_ctx *ctx, int S, int star, const double *x0, const double *goal, const double *goal_th,
                                   const double *region_g, const double *region_s, const double *sample_off,
                                   const double *ratial, double bi, int max_iter, const double *rnd, int nrnd, double *routes,
                                   int *route_len, int *n_nodes, int *fail_out, int *rnd_used, double *tree_nodes,
                                   int *tree_parent, double *tree_total, double *ms_kernel) {
  int rc = check_rrt_call(ctx, "cfs_rrt_find_routes", S, max_iter, nrnd, x0, goal, goal_th,
                          region_g && region_s && sample_off && ratial, rnd, routes, route_len, n_nodes, fail_out, rnd_used);
  if (rc || S == 0) return rc;
  const size_t nj = ctx->nj, cap = (size_t)max_iter + 2;
  std::vector<double> params(4 * nj);  // the device form's params block
  const double *parts[4] = {region_g, region_s, sample_off, ratial};
  for (int p = 0; p < 4; ++p) memcpy(params.data() + p * nj, parts[p], sizeof(double) * nj);
  const bool tree = tree_nodes && tree_parent && tree_total;
  double *d_x0, *d_goal, *d_gth, *d_params, *d_rnd, *d_routes, *d_tn = nullptr, *d_tt = nullptr;
  int *d_len, *d_nn, *d_fail, *d_used, *d_tp = nullptr;
  Area ar(ctx);
  ar.in(d_x0, x0, nj * S).in(d_goal, goal, nj * S).in(d_gth, goal_th, nj * S).in(d_params, params.data(), 4 * nj)
      .in(d_rnd, rnd, (size_t)nrnd * S).out(d_routes, routes, nj * cap * S).out(d_len, route_len, S).out(d_nn, n_nodes, S)
      .out(d_fail, fail_out, S).out(d_used, rnd_used, S);
  if (tree) ar.out(d_tn, tree_nodes, nj * cap * S).out(d_tt, tree_total, cap * S).out(d_tp, tree_parent, cap * S);
  if ((rc = ar.upload())) return rc;
  CU(cudaEventRecord(ctx->ev_a, ctx->stream));
  if ((rc = rrt_dev(ctx, S, star, d_x0, d_goal, d_gth, d_params, bi, max_iter, d_rnd, nrnd, d_routes, d_len, d_nn, d_fail, d_used,
                    d_tn, d_tp, d_tt)))
    return rc;
  CU(cudaEventRecord(ctx->ev_b, ctx->stream));
  if ((rc = ar.download())) return rc;
  if (ms_kernel) {
    float ms = 0;
    cudaEventElapsedTime(&ms, ctx->ev_a, ctx->ev_b);
    *ms_kernel = ms;
  }
  return 0;
}

extern "C" int cfs_rrt_find_routes_device(cfs_ctx *ctx, int S, int star, const double *x0, const double *goal, const double *goal_th,
                                          const double *params, double bi, int max_iter, const double *rnd, int nrnd,
                                          double *routes, int *route_len, int *n_nodes, int *fail_out, int *rnd_used,
                                          int *route_len_or_fail, int sync) {
  int rc = check_rrt_call(ctx, "cfs_rrt_find_routes_device", S, max_iter, nrnd, x0, goal, goal_th, params != nullptr, rnd, routes,
                          route_len, n_nodes, fail_out, rnd_used);
  if (rc || S == 0) return rc;
  CU(cudaSetDevice(ctx->device));
  if ((rc = rrt_dev(ctx, S, star, x0, goal, goal_th, params, bi, max_iter, rnd, nrnd, routes, route_len, n_nodes, fail_out, rnd_used,
                    nullptr, nullptr, nullptr)))
    return rc;
  if (route_len_or_fail) CU(launch_route_len_or_fail(S, route_len, fail_out, route_len_or_fail, ctx->stream));
  if (sync) CU(cudaStreamSynchronize(ctx->stream));
  return 0;
}

extern "C" int cfs_get_stats(const cfs_ctx *ctx, cfs_stats *out) {
  if (!ctx || !out) return CFS_E_ARG;
  *out = ctx->stats;
  return 0;
}

extern "C" int cfs_get_iter_times(const cfs_ctx *ctx, double *grad_ms, double *qp_ms, int cap) {
  if (!ctx) return CFS_E_ARG;
  int cnt = (int)ctx->it_grad_ms.size();
  if (cnt > cap) cnt = cap;
  for (int k = 0; k < cnt; ++k) {
    if (grad_ms) grad_ms[k] = ctx->it_grad_ms[k];
    if (qp_ms) qp_ms[k] = ctx->it_qp_ms[k];
  }
  return cnt;
}

extern "C" int cfs_get_qp_profile(cfs_ctx *ctx, long long *out8) {
  if (!ctx || !out8) return CFS_E_ARG;
  if (ctx->qpsteps.cap < sizeof(long long) * 32) return fail(ctx, CFS_E_STATE, "cfs_get_qp_profile: no solve yet");
  CU(cudaSetDevice(ctx->device));
  CU(cudaMemcpyAsync(out8, ptr<long long>(ctx->qpsteps) + 8, sizeof(long long) * 16, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return 0;
}

extern "C" int cfs_get_warp_profile(cfs_ctx *ctx, long long *out4) {
  if (!ctx || !out4) return CFS_E_ARG;
  out4[4] = ctx->last_warp_grid_warps;
  out4[5] = ctx->last_sms;
  if (ctx->qpsteps.cap < sizeof(long long) * 32) return fail(ctx, CFS_E_STATE, "cfs_get_warp_profile: no solve yet");
  CU(cudaSetDevice(ctx->device));
  CU(cudaMemcpyAsync(out4, ptr<long long>(ctx->qpsteps) + 24, sizeof(long long) * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return 0;
}

extern "C" int cfs_get_problem_steps(cfs_ctx *ctx, int *steps, int B) {
  if (!ctx || !steps || B < 0) return CFS_E_ARG;
  if ((size_t)B * sizeof(int) > ctx->probsteps.cap) return fail(ctx, CFS_E_ARG, "cfs_get_problem_steps: B exceeds the last batch");
  CU(cudaSetDevice(ctx->device));
  CU(cudaMemcpyAsync(steps, ctx->probsteps.p, sizeof(int) * B, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return 0;
}

extern "C" int cfs_set_option(cfs_ctx *ctx, const char *name, int value) {
  if (!ctx || !name) return CFS_E_ARG;
  if (strcmp(name, "fused") == 0) {
    ctx->use_fused = value != 0;
    return 0;
  }
  if (strcmp(name, "esc_steps") == 0) {
    ctx->esc_steps = value > 0 ? value : 0x7fffffff;
    return 0;
  }
  if (strcmp(name, "heavy_grid") == 0) { ctx->heavy_grid = value; return 0; }
  if (strcmp(name, "bulk_grid") == 0) { ctx->bulk_grid = value; return 0; }
  if (strcmp(name, "heavy_prio") == 0) { ctx->heavy_prio = value; return 0; }
  if (strcmp(name, "lpt") == 0) { ctx->lpt = value; return 0; }
  if (strcmp(name, "warp") == 0) { ctx->use_warp = value; return 0; }
  if (strcmp(name, "screen") == 0) { ctx->screen = value; return 0; }
  if (strcmp(name, "one_shot") == 0) { ctx->one_shot = value; return 0; }
  if (strcmp(name, "warp_lockstep") == 0) { ctx->use_warp_lockstep = value; return 0; }
  if (strcmp(name, "heavy_cfg") == 0) { ctx->heavy_cfg = value; return 0; }
  if (strcmp(name, "heavy_skip") == 0) { ctx->heavy_skip = value; return 0; }
  if (strcmp(name, "warp_cfg") == 0) { ctx->warp_cfg = value; return 0; }
  if (strcmp(name, "warp_zs") == 0) { ctx->warp_zs = value; return 0; }
  if (strcmp(name, "warp_qcap") == 0) { ctx->warp_qcap = value; return 0; }
  return fail(ctx, CFS_E_ARG, "cfs_set_option: unknown option '%s'", name);
}

extern "C" int cfs_set_timing(cfs_ctx *ctx, int level) {
  if (!ctx) return CFS_E_ARG;
  ctx->timing_level = level;
  return 0;
}

extern "C" int cfs_measure_fp64_peak(cfs_ctx *ctx, double *tflops, double *sm_clock_mhz_est) {
  if (!ctx || !tflops) return CFS_E_ARG;
  CU(cudaSetDevice(ctx->device));
  int sms = 0;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device);
  int rc;
  if ((rc = ensure(ctx, ctx->scratch_out, 64))) return rc;
  const int iters = 1 << 16, block = 256, grid = sms * 8;
  cudaStream_t st = ctx->stream;
  CU(launch_fp64_peak(ptr<double>(ctx->scratch_out), 1 << 12, grid, block, st));  // warm-up
  double best = 0;
  for (int rep = 0; rep < 5; ++rep) {
    CU(cudaEventRecord(ctx->ev_a, st));
    CU(launch_fp64_peak(ptr<double>(ctx->scratch_out), iters, grid, block, st));
    CU(cudaEventRecord(ctx->ev_b, st));
    CU(cudaStreamSynchronize(st));
    float ms = 0;
    cudaEventElapsedTime(&ms, ctx->ev_a, ctx->ev_b);
    const double fl = 2.0 * 8.0 * (double)iters * block * (double)grid;
    const double tf = fl / (ms * 1e-3) / 1e12;
    if (tf > best) best = tf;
  }
  *tflops = best;
  if (sm_clock_mhz_est) *sm_clock_mhz_est = best * 1e12 / (2.0 * 64.0 * sms) / 1e6;  // 64 FP64 FMA lanes per SM
  return 0;
}
