// k_fused.cu -- the whole CFS outer loop of one problem inside one persistent CTA (sm_100a).
//
// Replaces CFS_FANUC.optimizer (Lib/CFS_FANUC.m:62-79) end to end for the class path (num_jac gradients):
//   while ~stop_outer:  get_con (:101-135)  ->  Solve_QP (:83-98: quadprog + roll-out)  ->  EVAL (Lib/EVAL.m:51-73)
//
// Why fused (B200-first, not a translation of the MATLAB loop):
//   * the lock-step form (one K1 + one K3 launch per outer iteration over the still-active problems) pays, in every
//     iteration, for the slowest QP of that iteration while >90 % of the SMs idle (ncu: smsp__cycles_active 7 % of
//     elapsed in iteration 1).  Here every CTA carries ONE problem through ALL its outer iterations and then pulls the
//     next problem from a device work queue, so the batch costs max(longest single problem, total work / resident CTAs);
//   * the trajectory x_, the controls u, the linearised rows (-grad, rhs) and the QP working set never leave shared
//     memory between iterations: HBM sees each problem's inputs once and its outputs once (6.1 KB in, 6.3 KB out at
//     H = 50), the batch-shared Gram operator G (4.5 MB) streams from L2;
//   * the robot/obstacle tables are staged once per CTA with one TMA bulk copy (UBLKCP); the sin/cos values, kinematic
//     prefixes and running minima of a trajectory's num_jac evaluations (cfs_numjac_cols.cuh: 35 link steps per waypoint
//     instead of 55) live in shared memory that the QP phase reuses for its cached directions and working-set inverse;
//   * two tiers of the same code: the bulk tier (128 threads, 3 CTAs/SM, working sets of up to 15 rows with every member's
//     direction QQ^-1 c' cached in shared memory: no L2 access inside a dual step) hands the rare QP whose working set
//     outgrows that, or that needs more than esc_steps dual steps (almost always an infeasible linearisation on its way to
//     the infeasibility certificate), to the heavy tier (256 threads, 1 CTA/SM, 144 x 144 inverse on chip, primal recovery
//     through the Gram operator), which resumes the problem from its last completed outer iteration;
//   * the bulk tier pulls the problems longest-expected-first (launch_work_order, k_grad.cu): the ones whose reference line
//     passes inside an obstacle margin start first, so the batch ends with short problems instead of a tail of long ones.
#include "cfs_numjac_cols.cuh"
#include "qp_core.cuh"

namespace cfs {

#ifdef PF_GRAD_DETAIL
#define PF_GRAD(k) PF_ADD(k)
#define PF_ROWS 4
#else
#define PF_GRAD(k) do { } while (0)
#define PF_ROWS 0
#endif

#define FUSED_BULK_NT 128
#define FUSED_BULK_QS 16
#define FUSED_BULK_QZ 16  // cached directions: working sets of up to 15 rows + the candidate stay entirely in shared memory
#define FUSED_HEAVY_NT 256
#define FUSED_HEAVY_QS 144

struct FusedLayout {
  size_t qp_bytes, xs, us, tab, mbar, total;
};

__host__ __device__ inline FusedLayout fused_layout(int n, int nj, int OH, int m, int qs, int nt, int qz, bool lim = false) {
  FusedLayout L;
  size_t off[QP_NOFF];
  L.qp_bytes = qp_smem_layout(n, nj, OH, m, off, qs, nt, qz, lim);
  size_t o = L.qp_bytes;
  L.xs = o; o += sizeof(double) * 2 * n;
  L.us = o; o += sizeof(double) * n;
  o = (o + 127) / 128 * 128;
  L.tab = o; o += sizeof(DevTables);
  L.mbar = o; o += 16;
  L.total = (o + 15) / 16 * 16;
  return L;
}

// OFF: the obstacle rows read a.margin_off (per-waypoint margin offsets of the checked solve); a separate instantiation, the one
// without it is unchanged.  LIM (only with OFF): the QP also has the joint position rows of a.qlim.
template <int NJ, int NT, int QS, int MINB, int QZ, int MAXREG = (MINB == 1 ? 255 : 168), bool OFF = false, bool LIM = false>
__global__ void __launch_bounds__(NT) __maxnreg__(MAXREG) k_cfs_fused(SolveArgs a) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int n = a.n, nj = NJ, H = a.H, np = 3 * n, OH = a.nobs * H, m = OH + (LIM ? 6 : 4) * n, N = 2 * n;
  const int tid = threadIdx.x;
  const FusedLayout L = fused_layout(n, nj, OH, m, QS, NT, QZ, LIM);
  const QpView s = qp_view(smem_raw, n, nj, OH, m, QS, NT, QZ, LIM);
  const bool heavy = a.tier == 1;
  double *xs = reinterpret_cast<double *>(smem_raw + L.xs);  // x_  (CFS_FANUC.m:55)
  double *us = reinterpret_cast<double *>(smem_raw + L.us);  // u   (CFS_FANUC.m:56)
  DevTables &tab = *reinterpret_cast<DevTables *>(smem_raw + L.tab);
  uint64_t *mbar = reinterpret_cast<uint64_t *>(smem_raw + L.mbar);
  // gradient-phase scratch (sin/cos cache, f(x+-), kinematic prefixes, running minima): aliases the QP scratch span,
  // which starts at offset 0 of the layout
  const NumjacScratch nw = numjac_scratch(reinterpret_cast<double *>(smem_raw), NJ, H, OH);
  double *fv = nw.fv;  // f(x+), f(x-) per (obstacle, waypoint, column): [OH][NJ][2]

  tma_stage(&tab, a.tab, tab_bytes(a.nobs), mbar);
  const double *__restrict__ G = a.G;
  const int has_vel = a.has_lim, has_bnd = a.has_bounds;
#pragma unroll 1
  for (int e = tid; e < 3 * n; e += NT) s.gns[e] = a.gdiag[e] * a.gdiag[e];  // G_ii
#pragma unroll 1
  for (int e = tid; e < n; e += NT) s.ums[e] = has_bnd ? a.max_input[e] : 0.0;
  const double dt = tab.dt;
  const int ldg = a.slab_ld;
  double *Mgl = a.slab + (size_t)blockIdx.x * ldg * ldg;
  const QpDims dims = {n, nj, H, np, OH, m, has_vel, has_bnd, G, s.ums, Mgl, ldg, dt};
  const double qnan = __longlong_as_double(0x7ff8000000000000LL);
  long long steps_total = 0;
  int qmax_seen = 0;
  long long pf[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  long long tck = 0;
  const bool prof = a.prof != nullptr;

  const int count = heavy ? *a.esc_count : a.B;
  for (;;) {
    __syncthreads();
    if (tid == 0) s.ctl[0] = atomicAdd(heavy ? a.work_counter2 : a.work_counter, 1);
    __syncthreads();
    const int slot = s.ctl[0];
    if (slot >= count) break;
    const int b = heavy ? a.esc_list[slot] : (a.order ? a.order[slot] : slot);
    const double *x0 = a.x0 + (size_t)b * 2 * nj;
    const double *v0 = a.v0 + (size_t)b * np;

    // ---- problem set-up: u = 0, x_ = sys_info.x_, histories NaN, first stop test against x_old = ones (EVAL.m:47) ----
    PF_START();
    double part = 0.0;
    if (!heavy) {
#pragma unroll 1
      for (int e = tid; e < N; e += NT) {
        const double xv = a.xref[(size_t)b * N + e];
        xs[e] = xv;
        part += (xv - 1.0) * (xv - 1.0);
      }
#pragma unroll 1
      for (int e = tid; e < n; e += NT) us[e] = 0.0;
#pragma unroll 1
      for (int e = tid; e < a.max_outer; e += NT) {
        a.cost_hist[(size_t)b * a.max_outer + e] = qnan;
        if (a.e_u_hist) a.e_u_hist[(size_t)b * a.max_outer + e] = qnan;
      }
    } else {  // resume from the last completed outer iteration (written by the bulk tier)
#pragma unroll 1
      for (int e = tid; e < N; e += NT) xs[e] = a.x[(size_t)b * N + e];
#pragma unroll 1
      for (int e = tid; e < n; e += NT) us[e] = a.u[(size_t)b * n + e];
    }
#pragma unroll 1
    for (int pi = tid; pi < np; pi += NT) s.v0s[pi] = v0[pi];
    if (tid < 8) {
      s.lim[tid] = (tid < nj && has_vel) ? a.lim[tid] : 0.0;
      s.w0[tid] = (tid < nj) ? x0[nj + tid] : 0.0;
      if (LIM) {  // qmax | qmin | theta0 of the joint position rows
        s.lim[8 + tid] = (tid < nj) ? a.qlim[tid] : 0.0;
        s.lim[16 + tid] = (tid < nj) ? a.qlim[nj + tid] : 0.0;
        s.lim[24 + tid] = (tid < nj) ? x0[tid] : 0.0;
      }
    }
    const double nrm0 = sqrt(block_sum<NT>(part, s.red));
    const double cost0 = a.cost0[b];
    const double fupper = (has_bnd && a.fupper) ? a.fupper[b] : INFINITY;
    int status = -1, iters = 0, touched = 0, steps_prob = 0;
    if (heavy) {
      iters = a.iters[b];
      touched = (tid == 0) ? (a.status[b] & 0x100) : 0;
      steps_prob = a.prob_steps ? a.prob_steps[b] : 0;
    } else if (nrm0 < a.eps_outer) {
      status = 0;
    } else if (1 > a.max_outer) {
      status = 1;
    }
    PF_ADD(0);
    pf[6] += 1;

    for (int it = iters + 1; status < 0; ++it) {
      // ---- get_con: distances + num_jac gradients of every waypoint, rows written in place (CFS_FANUC.m:110-124) ----
      PF_START();
      __syncthreads();  // the sin/cos cache aliases the previous QP's scratch
      numjac_sincos<NJ, NT>(tab, xs, H, nw.scw);
      __syncthreads();
      PF_GRAD(1);
      // pass 1: one thread per waypoint runs the all-minus chain M_i and the base chain B_i side by side;
      // pass 2: NJ*H items of NJ link steps (P_t then N_{NJ-1-t} from M's stored prefixes), two per thread
#pragma unroll 1
      for (int pass = 1; pass <= 2; ++pass) {
        const int items = pass == 1 ? H : NJ * H;
        const int stride = pass == 1 ? NT : 2 * NT;
#pragma unroll 1
        for (int eA = tid; eA < items; eA += stride) {
          bool hasB = true;
          int iA = eA, tyA = 1, iB = eA, tyB = 0;
          if (pass == 2) {
            hasB = eA + NT < items;
            const int eB = hasB ? eA + NT : eA;
            tyA = eA / H;
            iA = eA - tyA * H;
            tyB = eB / H;
            iB = eB - tyB * H;
          }
#pragma unroll 1
          for (int j0 = 0; j0 < a.nobs; j0 += 2)
            numjac_items2<NJ>(tab, nw, H, pass, iA, tyA, iB, tyB, hasB, j0, a.nobs, touched, s.orhs);
        }
        __syncthreads();
        PF_GRAD(1 + pass);
      }
#pragma unroll 1
      for (int cid = tid; cid < OH; cid += NT) {  // I = distance - margin (CFS_FANUC.m:117)
        const int j = cid / H;
        const double margin = a.margin_is_D ? tab.obs[j].D : tab.obs[j].eps;
        s.orhs[cid] -= OFF ? margin + a.margin_off[(size_t)b * OH + cid] : margin;
      }
      __syncthreads();
#pragma unroll 1
      for (int e = tid; e < OH * NJ; e += NT)  // l = -Diff'*Bj(1:njoint,:) (:121), Diff = (yhi - ylo)/eps (num_jac.m:15)
        s.ocoef[e] = -((fv[2 * e] - fv[2 * e + 1]) / CFS_NUMJAC_EPS);
      __syncthreads();
      if (it > 1)  // s = I - Diff'*Bj*u (:120); B_theta u = theta_i - (theta_0 + i dt w_0) once x_ is the roll-out of u
#pragma unroll 1
        for (int cid = tid; cid < OH; cid += NT) {
          const int i = cid % H;
          double gu = 0.0;
#pragma unroll
          for (int k = 0; k < NJ; ++k)
            gu += -s.ocoef[cid * NJ + k] * (xs[i * 2 * NJ + k] - (x0[k] + ((i + 1) * dt) * x0[NJ + k]));
          s.orhs[cid] -= gu;
        }
      __syncthreads();
#pragma unroll 1
      for (int pi = tid; pi < np; pi += NT) s.v[pi] = s.v0s[pi];
#pragma unroll 1
      for (int e = tid; e < m; e += NT) s.inact[e] = 0;
#pragma unroll 1
      for (int cid = tid; cid < OH; cid += NT) {
        const int i = wp_of(cid, H);
        double sg = 0.0;
#pragma unroll
        for (int k = 0; k < NJ; ++k) sg += s.ocoef[cid * NJ + k] * s.ocoef[cid * NJ + k] * s.gns[i * NJ + k];
        s.onrm[cid] = sg;  // scan normalisation (diagonal proxy of c QQ^-1 c')
      }
      if (tid == 0) s.toff[0] = 0;
      __syncthreads();
      PF_ADD(PF_ROWS);

      // ---- Solve_QP (CFS_FANUC.m:85) ----
      int q = 0, steps = 0;
      const int masked = qp_mask_antiparallel<NT>(s, dims);
      const int qst = qp_solve<NT, QS, (MINB == 1), NJ, QZ, LIM>(s, dims, cost0, fupper, false, q, steps, qmax_seen, pf, tck, prof,
                                                        heavy ? 0x7fffffff : a.esc_steps, masked);
      steps_total += steps;
      steps_prob += steps;
      if (qst != 0) {  // 2 infeasible / 3 numerical: u, x_ keep the previous iterate; 4: the heavy tier redoes this iteration
        status = qst;
        break;
      }
      // ---- e_u, cost by duality, roll-out, stop rule (EVAL.m:51-73, CFS_FANUC.m:88-94) ----
      double pe = 0.0;
#pragma unroll 1
      for (int c = tid; c < n; c += NT) {
        const double un = s.v[2 * n + c];
        const double dlt = us[c] - un;
        pe += dlt * dlt;
        us[c] = un;
      }
      const double e_u = sqrt(block_sum<NT>(pe, s.red));
      double pc = 0.0;
#pragma unroll 1
      for (int w = tid; w < q; w += NT) pc -= s.lam[w] * slack_at<NJ, LIM>(s.act[w], dims, s, s.v0s);
      const double cost = cost0 + 0.5 * block_sum<NT>(pc, s.red);
      double px = 0.0;
      if (tid < nj) {
        double th = x0[tid], om = x0[nj + tid];
        for (int i = 0; i < H; ++i) {
          const double uk = us[i * nj + tid];
          const double thn = (th + dt * om) + (0.5 * dt * dt) * uk;
          const double omn = om + dt * uk;
          th = thn;
          om = omn;
          double *xr = xs + (size_t)i * 2 * nj;
          const double d1 = th - xr[tid], d2 = om - xr[nj + tid];
          px += d1 * d1 + d2 * d2;
          xr[tid] = th;
          xr[nj + tid] = om;
        }
      }
      const double dx = sqrt(block_sum<NT>(px, s.red));
      if (tid == 0) {
        a.cost_hist[(size_t)b * a.max_outer + (it - 1)] = cost;
        if (a.e_u_hist) a.e_u_hist[(size_t)b * a.max_outer + (it - 1)] = e_u;
      }
      iters = it;
      if (dx < a.eps_outer)
        status = 0;  // converged (EVAL.m:64-67)
      else if (it + 1 > a.max_outer)
        status = 1;  // MAX_ITER (EVAL.m:69-72)
      PF_ADD(5);
    }

    // ---- results ----
    __syncthreads();
#pragma unroll 1
    for (int e = tid; e < n; e += NT) a.u[(size_t)b * n + e] = us[e];
#pragma unroll 1
    for (int e = tid; e < N; e += NT) a.x[(size_t)b * N + e] = xs[e];
    const int any_touch = __syncthreads_or(touched);
    if (tid == 0) {
      a.iters[b] = iters;
      a.status[b] = status | (any_touch ? 0x100 : 0);
      if (a.prob_steps) a.prob_steps[b] = steps_prob;
      if (status == 4) a.esc_list[atomicAdd(a.esc_count, 1)] = b;
    }
  }
  if (prof && tid == 0)
    for (int k = 0; k < 8; ++k)
      if (pf[k]) atomicAdd(reinterpret_cast<unsigned long long *>(a.prof + (heavy ? 8 : 0) + k), (unsigned long long)pf[k]);
  if (tid == 0) {
    if (steps_total) atomicAdd(reinterpret_cast<unsigned long long *>(a.qp_steps), (unsigned long long)steps_total);
    if (qmax_seen) atomicMax(a.max_active, qmax_seen);
  }
}

static bool fused_supported_nj(int nj) { return nj == 2 || nj == 5; }

// tier 0: bulk (CTA per problem); tier 1: heavy, 144 x 144 inverse on chip (a whole SM per CTA); tier 2: "slim" heavy,
// FUSED_SLIM_QS^2 on chip and the rest spilled to the global slab, 168 registers: leaves room for bulk warps on the same SM
#define FUSED_SLIM_QS 64
static void tier_cfg(int tier, int &nt, int &qs, int &qz) {
  nt = tier ? FUSED_HEAVY_NT : FUSED_BULK_NT;
  qs = tier == 2 ? FUSED_SLIM_QS : (tier ? FUSED_HEAVY_QS : FUSED_BULK_QS);
  qz = tier ? 0 : FUSED_BULK_QZ;
}

size_t fused_smem_bytes(const SolveArgs &a, int tier) {
  int nt, qs, qz;
  tier_cfg(tier, nt, qs, qz);
  const int OH = a.nobs * a.H;
  const bool lim = a.qlim != nullptr;
  return fused_layout(a.n, a.nj, OH, OH + (lim ? 6 : 4) * a.n, qs, nt, qz, lim).total;
}

bool fused_supported(const SolveArgs &a) {
  if (!fused_supported_nj(a.nj)) return false;
  const int OH = a.nobs * a.H;
  for (int tier = 0; tier < 3; ++tier) {
    int nt, qs, qz;
    tier_cfg(tier, nt, qs, qz);
    // the gradient-phase scratch must fit into the QP scratch span it aliases, and the CTA into one SM's shared memory
    (void)nt;
    if (sizeof(double) * numjac_scratch_doubles(a.nj, a.H, OH) > qp_scratch_span(a.n, a.nj, OH, qs, qz)) return false;
    if (fused_smem_bytes(a, tier) > 227 * 1024) return false;
  }
  return true;
}

template <class K>
static int grid_of(K kernel, int nt, size_t smem, int device) {
  int sms = 0, per = 0;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
  // the opt-in maximum, not this configuration's size: the attribute is per function and shared by every context of the process
  if (smem > 227 * 1024 || cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) != cudaSuccess) return 0;
  cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per, kernel, nt, smem);
  return sms * per;
}

typedef void (*FusedKernel)(SolveArgs);
template <int NJ, bool OFF, bool LIM = false>
static FusedKernel fused_kernel_nj(int tier) {
  if (tier == 0) return k_cfs_fused<NJ, FUSED_BULK_NT, FUSED_BULK_QS, 3, FUSED_BULK_QZ, 168, OFF, LIM>;
  if (tier == 1) return k_cfs_fused<NJ, FUSED_HEAVY_NT, FUSED_HEAVY_QS, 1, 0, 255, OFF, LIM>;
  return k_cfs_fused<NJ, FUSED_HEAVY_NT, FUSED_SLIM_QS, 1, 0, 168, OFF, LIM>;
}
// tier 0 bulk, 1 heavy, 2 slim heavy; the margin-offset instantiations when a.margin_off is set, the joint-limit ones (which
// also read the offsets) when a.qlim is set
static FusedKernel fused_kernel(const SolveArgs &a, int tier) {
  const bool off = a.margin_off != nullptr, lim = a.qlim != nullptr;
  if (lim && !off) return nullptr;
  if (a.nj == 2) return lim ? fused_kernel_nj<2, true, true>(tier) : (off ? fused_kernel_nj<2, true>(tier) : fused_kernel_nj<2, false>(tier));
  if (a.nj == 5) return lim ? fused_kernel_nj<5, true, true>(tier) : (off ? fused_kernel_nj<5, true>(tier) : fused_kernel_nj<5, false>(tier));
  return nullptr;
}

int fused_max_grid(const SolveArgs &a, int device, int tier) {
  FusedKernel k = fused_kernel(a, tier);
  if (!k) return 0;
  return grid_of(k, tier == 0 ? FUSED_BULK_NT : FUSED_HEAVY_NT, fused_smem_bytes(a, tier), device);
}

cudaError_t launch_fused(const SolveArgs &a_in, int grid, int tier, cudaStream_t st) {
  SolveArgs a = a_in;
  a.tier = tier ? 1 : 0;
  FusedKernel k = fused_kernel(a, tier);
  if (!k) return cudaErrorInvalidValue;
  k<<<grid, tier == 0 ? FUSED_BULK_NT : FUSED_HEAVY_NT, fused_smem_bytes(a, tier), st>>>(a);
  return cudaGetLastError();
}

}  // namespace cfs
