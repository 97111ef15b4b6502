// k_check.cu -- continuous collision checks of joint-space edges and CFS trajectory segments, sm_100a, FP64.
//
// The reference only checks configurations (RRT_FANUC.m:146-181 checks the nodes, CFS_FANUC.get_con constrains the
// waypoints); these kernels certify the arm along the whole path between two configurations.  Semantics in
// include/cfs_b200.h (cfs_check_edges / cfs_check_trajectories); the CPU restatement is tests/check_oracle.c.
//
// Clearance c(theta) = min over links l and obstacles j of (d_lj(theta) - m_j), with the same FK (xf_first / xf_step_inplace /
// link_endpoints) and the same link-axis distance (link_obs_key, touch rule included) as every other kernel.  Conservative
// advancement: |c(theta1) - c(theta2)| <= sum_j R_j TV_j, so from a point with clearance c the path stays above -eta for
// (c + eta) / vmax more units of its parameter.  One item (an edge, or one segment of a trajectory) is one thread; the
// number of evaluations per item is heavy-tailed (1 .. ~1500), so the grid is persistent and every lane that finishes
// pulls the next item at once (warp-aggregated atomics on one counter) instead of idling until its warp is done.
#include "cfs_geom.cuh"
#include "cfs_kernels.cuh"

namespace cfs {

#define CHK_THREADS 128

// c(theta): the minimum over (link, obstacle) of the signed distance minus the margin.  sqrt and "- m_j" are monotone, so this
// equals min_j (min_l d_lj - m_j) and, with one obstacle, RN(dmin - D) of k_nodes_feasible bit for bit.
template <int NJ>
__device__ __forceinline__ double clearance(const DevTables &tab, const double th[NJ], int nobs, int margin_is_D) {
  Xf M;
  double p[6];
  int touched = 0;
  double c = INFINITY;
#pragma unroll
  for (int l = 0; l < NJ; ++l) {
    double sn, cs;
    sincos(th[l] + tab.link[l].th_off, &sn, &cs);
    if (l == 0)
      xf_first(tab.link[0], cs, sn, M);
    else
      xf_step_inplace(M, tab.link[l], cs, sn);
    link_endpoints(M, tab.link[l], tab.base, p);
#pragma unroll 1
    for (int j = 0; j < nobs; ++j) {
      const ObsTab &o = tab.obs[j];
      const double v = key_to_dist(link_obs_key(p, o, touched)) - (margin_is_D ? o.D : o.eps);
      c = v < c ? v : c;
    }
  }
  return c;
}

// MODE 0: edges theta(s) = a + s (b - a), s in [0, 1].  MODE 1: segment k of trajectory b, theta(tau) = theta_k + omega_k tau +
// (0.5 tau^2) u_k, tau in [0, dt].  Path, step and vmax are written with explicit round-to-nearest operations (no FMA
// contraction): the same operations in the same order as the CPU restatement.
// Start of item `it` and the derivative of its path: edges a, b - a; segments theta_k, omega_k, u_k (x0 for k = 0).
template <int NJ, int MODE>
__device__ __forceinline__ void item_ptrs(const CheckArgs &a, int it, const double *&p0, const double *&p1, const double *&pu) {
  if (MODE == 0) {
    p0 = a.theta_a + (long long)it * NJ;
    p1 = a.theta_b + (long long)it * NJ;
    pu = nullptr;
  } else {
    const int b = it / a.H, k = it - b * a.H;
    p0 = k == 0 ? a.x0 + (long long)b * 2 * NJ : a.x + ((long long)b * a.H + (k - 1)) * 2 * NJ;
    p1 = p0 + NJ;
    pu = a.u + ((long long)b * a.H + k) * NJ;
  }
}

// MODE 0: edges theta(s) = a + s (b - a), s in [0, 1].  MODE 1: segment k of trajectory b, theta(tau) = theta_k + omega_k tau +
// (0.5 tau^2) u_k, tau in [0, dt].  Path, step and vmax are written with explicit round-to-nearest operations (no FMA
// contraction): the same operations in the same order as the CPU restatement.  A lane keeps only its item's scalars in
// registers and re-reads the item's inputs (L1-resident) at every evaluation: nothing stays live across the out-of-line box
// distance, and a cap of 168 registers (instead of __launch_bounds__, whose choice of 128 spilled the nj = 2 segment form around
// that call): no instantiation spills.  The 80-byte stack frame is sincos's argument reduction, as in every FK kernel.
template <int NJ, int MODE>
__global__ void __maxnreg__(168) k_check(CheckArgs a) {
  __shared__ alignas(128) DevTables tab;
  __shared__ alignas(8) uint64_t mbar;
  tma_stage(&tab, a.tab, tab_bytes(a.nobs), &mbar);
  const int lane = threadIdx.x & 31;
  const double dt = tab.dt, half_eta = 0.5 * a.eta;
  double s = 0.0, send = 0.0, vmax = 0.0, cmin = INFINITY;
  int item = -1, ev = 0;
  bool more = true;
  for (;;) {
    // lanes without an item take the next ones: one atomic per warp, consecutive items per lane
    const bool need = item < 0 && more;
    const unsigned m = __ballot_sync(0xffffffffu, need);
    if (m) {
      const int leader = __ffs(m) - 1;
      int base = 0;
      if (lane == leader) base = atomicAdd(a.counter, __popc(m));
      base = __shfl_sync(0xffffffffu, base, leader);
      if (need) {
        const int it = base + __popc(m & ((1u << lane) - 1u));
        if (it < a.N) {
          const double *p0, *p1, *pu;
          item_ptrs<NJ, MODE>(a, it, p0, p1, pu);
          item = it;
          s = 0.0;
          cmin = INFINITY;
          ev = 0;
          vmax = 0.0;
#pragma unroll
          for (int k = 0; k < NJ; ++k) {
            double w;
            if (MODE == 0) {
              w = fabs(__dsub_rn(__ldg(p1 + k), __ldg(p0 + k)));
            } else {
              const double om = __ldg(p1 + k);
              const double w0 = fabs(om), w1 = fabs(__dadd_rn(om, __dmul_rn(__ldg(pu + k), dt)));
              w = w0 > w1 ? w0 : w1;
            }
            vmax = __dadd_rn(vmax, __dmul_rn(a.R[k], w));
          }
          send = MODE == 0 ? 1.0 : dt;
        } else {
          more = false;
        }
      }
    }
    if (!__any_sync(0xffffffffu, item >= 0)) break;
    if (item < 0) continue;
    int verdict = -1;
    double hit_at = -1.0;
    if (ev == a.max_evals) {
      verdict = CHK_UNDECIDED;
    } else {
      const double *p0, *p1, *pu;
      item_ptrs<NJ, MODE>(a, item, p0, p1, pu);
      double th[NJ];
#pragma unroll
      for (int k = 0; k < NJ; ++k) {
        const double t0 = __ldg(p0 + k);
        th[k] = MODE == 0 ? __dadd_rn(t0, __dmul_rn(s, __dsub_rn(__ldg(p1 + k), t0)))
                          : __dadd_rn(__dadd_rn(t0, __dmul_rn(__ldg(p1 + k), s)), __dmul_rn(__dmul_rn(__dmul_rn(0.5, s), s), __ldg(pu + k)));
      }
      const double c = clearance<NJ>(tab, th, a.nobs, a.margin_is_D);
      ++ev;
      cmin = c < cmin ? c : cmin;
      if (c < -half_eta) {
        verdict = CHK_HIT;
        hit_at = s;
      } else if (s == send || vmax == 0.0) {
        verdict = CHK_CLEAR;
      } else {
        s = __dadd_rn(s, __ddiv_rn(__dadd_rn(c, a.eta), vmax));
        if (!(s < send)) s = send;
      }
    }
    if (verdict >= 0) {
      a.verdict[item] = verdict;
      a.s_hit[item] = hit_at;
      a.cmin[item] = cmin;
      if (a.evals) a.evals[item] = ev;
      item = -1;
    }
  }
}

// per trajectory, segments in order: HIT if any segment hits (t_hit = k dt + tau of the first one), else UNDECIDED if any is,
// else CLEAR; cmin = min, evals = sum.  A sequential pass per trajectory: the result does not depend on scheduling.
__global__ void k_check_reduce(int B, int H, double dt, const int *sv, const double *ss, const double *sc, const int *se,
                               int *verdict, double *t_hit, double *cmin, int *evals) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  int hit = 0, und = 0, ev = 0;
  double th = -1.0, cm = INFINITY;
  for (int k = 0; k < H; ++k) {
    const long long i = (long long)b * H + k;
    const int v = sv[i];
    if (v == CHK_HIT && !hit) {
      hit = 1;
      th = __dadd_rn(__dmul_rn((double)k, dt), ss[i]);
    }
    und |= v == CHK_UNDECIDED;
    cm = sc[i] < cm ? sc[i] : cm;
    ev += se[i];
  }
  verdict[b] = hit ? CHK_HIT : (und ? CHK_UNDECIDED : CHK_CLEAR);
  t_hit[b] = th;
  cmin[b] = cm;
  if (evals) evals[b] = ev;
}

template <int NJ, int MODE>
static cudaError_t launch_check_nj(const CheckArgs &a, int device, cudaStream_t s) {
  int sms = 0, per = 0;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
  cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per, k_check<NJ, MODE>, CHK_THREADS, 0);
  if (e != cudaSuccess) return e;
  long long grid = (long long)sms * (per > 0 ? per : 1);
  const long long need = ((long long)a.N + CHK_THREADS - 1) / CHK_THREADS;
  if (grid > need) grid = need;
  k_check<NJ, MODE><<<(int)grid, CHK_THREADS, 0, s>>>(a);
  return cudaGetLastError();
}

template <int MODE>
static cudaError_t launch_check_mode(const CheckArgs &a, int device, cudaStream_t s) {
  switch (a.nj) {
    case 2: return launch_check_nj<2, MODE>(a, device, s);
    case 3: return launch_check_nj<3, MODE>(a, device, s);
    case 4: return launch_check_nj<4, MODE>(a, device, s);
    case 5: return launch_check_nj<5, MODE>(a, device, s);
    case 6: return launch_check_nj<6, MODE>(a, device, s);
    default: return cudaErrorInvalidValue;
  }
}

cudaError_t launch_check(const CheckArgs &a, int device, cudaStream_t s) {
  if (a.N <= 0) return cudaSuccess;
  cudaError_t e = cudaMemsetAsync(a.counter, 0, sizeof(int), s);
  if (e != cudaSuccess) return e;
  return a.mode == 0 ? launch_check_mode<0>(a, device, s) : launch_check_mode<1>(a, device, s);
}

cudaError_t launch_check_reduce(int B, int H, double dt, const int *sv, const double *ss, const double *sc, const int *se,
                                int *verdict, double *t_hit, double *cmin, int *evals, cudaStream_t s) {
  if (B <= 0) return cudaSuccess;
  k_check_reduce<<<(B + 127) / 128, 128, 0, s>>>(B, H, dt, sv, ss, sc, se, verdict, t_hit, cmin, evals);
  return cudaGetLastError();
}

}  // namespace cfs
