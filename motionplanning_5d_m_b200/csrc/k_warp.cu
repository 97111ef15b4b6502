// k_warp.cu -- bulk tier of the fused CFS solver: ONE WARP carries one problem through all its outer iterations (sm_100a).
//
// Replaces CFS_FANUC.optimizer (Lib/CFS_FANUC.m:62-79) end to end for the class path (num_jac gradients):
//   while ~stop_outer:  get_con (:101-135)  ->  Solve_QP (:83-98: quadprog + roll-out)  ->  EVAL (Lib/EVAL.m:51-73)
//
// Why a warp and not a CTA per problem (round-1 bulk tier, k_fused.cu, ncu r01: 2.7 warps per scheduler of which most wait at
// CTA barriers -- stall_barrier 21 %, H = 50 waypoints leave 78 of 128 threads idle in the first gradient pass, every block
// reduction costs two barriers): a problem-iteration is ~1750 link steps + a handful of O(n) QP phases, i.e. enough work
// for 32 lanes but not for 128.  With one warp per problem
//   * there is no CTA barrier at all: phases are separated by __syncwarp(), reductions are five shuffles;
//   * 9-12 problems are resident per SM, each an independent instruction stream (the gradient phase of one overlaps the
//     QP phase of another), instead of 3;
//   * shared memory per problem shrinks from 73.6 KB to ~18-22 KB: only theta, u, u0, the rows and the cached directions
//     stay on chip; omega / previous controls / x_ stream through L2 once per outer iteration; B_theta u and B_omega u
//     are recomputed by warp prefix sums instead of being stored (qp_warp.cuh);
//   * gradient phase: one lane = one waypoint (K1's prefix-sharing evaluation order, 35 link steps instead of 55), the
//     sin/cos cache and the kinematic prefix in lane-private shared-memory columns that alias the direction cache.
// The robot/obstacle tables are staged once per CTA by one TMA bulk copy (UBLKCP) and shared by its warps.
// Problems whose working set outgrows 15 rows, or that need more than esc_steps dual steps in one QP, are handed to the heavy
// tier (k_fused.cu, tier 1), which resumes them from their last completed outer iteration.
// One solve is several launches of this kernel (cfs_api.cu, "screening passes"): a launch with it_stop = k stops every problem
// after outer iteration k and appends the unfinished ones to a continuation list that the next launch resumes (phase 2), so
// that the heavy tier can start on the long dual chains of the early iterations while most of the work is still ahead.
#include "cfs_geom.cuh"
#include "qp_warp.cuh"

namespace cfs {

template <int NJ>
__device__ __forceinline__ void lane_sc(const double *sc, int lane, int l, int kind, double &c, double &s) {
  const double c0 = sc[(0 * NJ + l) * 32 + lane], s0 = sc[(1 * NJ + l) * 32 + lane];
  if (kind == 0) {
    c = c0;
    s = s0;
    return;
  }
  // angle addition with the correctly rounded cos / sin of eps/2 (cfs_types.cuh): same operations as numjac_sincos
  const double cc = c0 * CFS_NUMJAC_COSH, ss = s0 * CFS_NUMJAC_COSH;
  if (kind == 1) {  // theta + eps/2   (num_jac.m:11)
    c = fma(-s0, CFS_NUMJAC_SINH, cc);
    s = fma(c0, CFS_NUMJAC_SINH, ss);
  } else {  // theta - eps/2   (num_jac.m:13)
    c = fma(s0, CFS_NUMJAC_SINH, cc);
    s = fma(-c0, CFS_NUMJAC_SINH, ss);
  }
}

__device__ __forceinline__ double wmin_first(double cur, double cand) { return cand < cur ? cand : cur; }

// One waypoint of get_con's loop body (CFS_FANUC.m:113-118) on one lane: distance, linkid rule and num_jac gradient against
// obstacles j0 .. j0+OC-1.  Evaluation order of cfs_numjac.cuh (every evaluated value identical): num_jac never resets xp
// (num_jac.m:13-14), so column k is evaluated with joints < k at theta - eps/2; the 11 evaluations of a waypoint are 2 NJ + 1
// segments of one flat loop -- seg 0: y = f(x); seg 2k+1: yhi of column k (from the "all minus" prefix Mm_{k-1}: link k at
// theta + eps/2, links > k at theta); seg 2k+2: ylo of column k (link k at theta - eps/2, which also extends the prefix) --
// 35 link steps instead of 55, and ONE instance of the link-step body in the instruction stream (several warps of an SM are in
// different phases of different problems: the 32 KB instruction cache has to hold all of them).
// sc: [2][NJ][32] cos/sin at theta, pm: [12][32] running prefix; both lane-private shared-memory columns.
template <int NJ, int OC>
__device__ __forceinline__ void numjac_waypoint_lane(const DevTables &tab, const double *sc, double *pm, int lane, int j0,
                                                     int nobs, int &touched, double *dist_out, double *ocoef, int cid0,
                                                     int cid_stride) {
  double dpre[OC], yhi[OC];
#pragma unroll
  for (int jj = 0; jj < OC; ++jj) {
    dpre[jj] = INFINITY;
    yhi[jj] = 0.0;
  }
  Xf M;
#pragma unroll 1
  for (int seg = 0; seg <= 2 * NJ; ++seg) {
    const int k = seg == 0 ? 0 : (seg - 1) >> 1;
    const bool isP = seg & 1, isN = seg > 0 && !isP;
    double dcur[OC], dk[OC];
#pragma unroll
    for (int jj = 0; jj < OC; ++jj) {
      dcur[jj] = seg == 0 ? INFINITY : dpre[jj];
      dk[jj] = 0.0;
    }
#pragma unroll 1
    for (int l = k; l < NJ; ++l) {
      double c, s, p[6];
      lane_sc<NJ>(sc, lane, l, (seg > 0 && l == k) ? (isP ? 1 : 2) : 0, c, s);
      if (l == k) {  // segment start
        if (k == 0) {
          xf_first(tab.link[0], c, s, M);
        } else {
#pragma unroll
          for (int e = 0; e < 12; ++e) M.m[e] = pm[e * 32 + lane];
          xf_step_inplace(M, tab.link[k], c, s);
        }
        if (isN && k + 1 < NJ) {  // running prefix Mm_0 ... Mm_k
#pragma unroll
          for (int e = 0; e < 12; ++e) pm[e * 32 + lane] = M.m[e];
        }
      } else {
        xf_step_inplace(M, tab.link[l], c, s);
      }
      link_endpoints(M, tab.link[l], tab.base, p);
#pragma unroll
      for (int jj = 0; jj < OC; ++jj)
        if (j0 + jj < nobs) {
          const double key = link_obs_key(p, tab.obs[j0 + jj], touched);  // signed squares, see cfs_geom.cuh
          if (l == k) dk[jj] = key;
          dcur[jj] = wmin_first(dcur[jj], key);  // strict <: first minimal link (dist_arm_3D_Heu_2.m:25-28)
        }
    }
#pragma unroll
    for (int jj = 0; jj < OC; ++jj)
      if (j0 + jj < nobs) {
        const double val = key_to_dist(dcur[jj]);  // the only square root of this evaluation of dist_arm
        if (seg == 0) {
          dist_out[jj] = val;
        } else if (isP) {
          yhi[jj] = val;
        } else {
          // l = -Diff'*Bj(1:njoint,:) (CFS_FANUC.m:121), Diff(k) = (yhi - ylo)/eps (num_jac.m:15)
          ocoef[(size_t)(cid0 + jj * cid_stride) * NJ + k] = -((yhi[jj] - val) / CFS_NUMJAC_EPS);
          dpre[jj] = wmin_first(dpre[jj], dk[jj]);
        }
      }
  }
}

struct WarpSmem {
  size_t tab, mbar, regions, region_bytes, total;
};
__host__ __device__ inline WarpSmem warp_smem(int n, int nj, int OH, int zs, int wpc, int nobs, bool lim = false) {
  WarpSmem L;
  size_t o = 0;
  L.tab = o; o += CFS_TAB_HEADER_BYTES + sizeof(ObsTab) * (size_t)nobs;  // only the staged part of DevTables
  L.mbar = o; o += 16;
  o = (o + 127) / 128 * 128;
  L.regions = o;
  L.region_bytes = (warp_region_bytes(n, nj, OH, zs, lim) + 127) / 128 * 128;
  L.total = o + L.region_bytes * wpc;
  return L;
}

// PROF: clock64 split of every problem into gradient phase / QP / everything (timing level 3: cfs_get_warp_profile); a separate
// instantiation so that the production kernel keeps its register budget.  OFF: the obstacle rows read a.margin_off (the
// checked solve's per-waypoint margin offsets); also a separate instantiation, the one without it is unchanged.  LIM (only
// with OFF): the QP also has the joint position rows of a.qlim.
template <int NJ, int NT, int MAXREG, int OC, bool PROF = false, bool OFF = false, bool LIM = false>
__global__ void __launch_bounds__(NT) __maxnreg__(MAXREG) k_cfs_warp(SolveArgs a) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  constexpr int WPC = NT / 32;
  const int n = a.n, H = a.H, O = a.nobs, OH = O * H, m = OH + (LIM ? 6 : 4) * n, N = 2 * n;
  const int mz = LIM ? OH + 4 * n + (2 * n + 7) / 8 : m;  // bytes of the inact map (LIM: position rows as bits)
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const WarpSmem L = warp_smem(n, NJ, OH, a.warp_zs, WPC, O, LIM);
  DevTables &tab = *reinterpret_cast<DevTables *>(smem_raw + L.tab);
  uint64_t *mbar = reinterpret_cast<uint64_t *>(smem_raw + L.mbar);
  tma_stage(&tab, a.tab, tab_bytes(a.nobs), mbar);

  WView s = warp_view(smem_raw + L.regions + L.region_bytes * wid, n, NJ, OH, a.warp_zs);
  s.zgl = a.zslab + (size_t)(blockIdx.x * WPC + wid) * warp_slab_doubles(n, a.warp_zs);
  s.Mgl = s.zgl + (size_t)(WQ_QZ - a.warp_zs) * n;
  s.qcap = a.warp_qcap < WQ_QBIG - 1 ? (a.warp_qcap > 1 ? a.warp_qcap : 1) : WQ_QBIG - 1;
  double *sc = s.zc, *pm = s.zc + 2 * NJ * 32;  // gradient-phase scratch aliases the direction cache
  const double dt = tab.dt, dt2 = dt * dt;
  const WDims P = {n, H, OH, O, m, 3 * n, a.has_lim, a.has_bounds, dt, a.G, a.gdiag, a.max_input, a.lim, LIM ? a.qlim : nullptr};
  const double qnan = __longlong_as_double(0x7ff8000000000000LL);
  long long steps_total = 0;
  int qmax_seen = 0;
  long long pf_grad = 0, pf_qp = 0, pf_all = 0, pf_passes = 0, pf_t0 = 0, pf_t1 = 0;

  const bool resume = a.phase == 2;
  const int count = resume ? *a.cont_count : a.B;
  for (int round = 0;; ++round) {
    int slot = 0;
    if (a.one_shot) {  // one problem per warp, then the CTA leaves the SM (see cfs_set_option "one_shot")
      if (round > 0) break;
      slot = blockIdx.x * WPC + wid;
    } else {
      if (lane == 0) slot = atomicAdd(a.work_counter, 1);
      slot = __shfl_sync(FULLMASK, slot, 0);
    }
    if (slot >= count) break;
    const int b = resume ? a.cont_list[slot] : (a.order ? a.order[slot] : slot);
    const double *x0 = a.x0 + (size_t)b * 2 * NJ;
    const double *xref = a.xref + (size_t)b * N;
    double *ub = a.u + (size_t)b * n;
    double *xb = a.x + (size_t)b * N;
    if (PROF) pf_t0 = clock64();

    // ---- problem set-up: u = 0, x_ = sys_info.x_, histories NaN, first stop test against x_old = ones (EVAL.m:47) ----
    __syncwarp();
    double part = 0.0;
#pragma unroll 2
    for (int e = lane; e < N; e += 32) {
      const double xv = resume ? xb[e] : xref[e];  // resume: x_ of the completed iterations
      part += (xv - 1.0) * (xv - 1.0);
      if (!resume) xb[e] = xv;
      const int i = e / (2 * NJ), r = e - i * 2 * NJ;
      if (r < NJ) s.th[i * NJ + r] = xv;
    }
#pragma unroll 2
    for (int c = lane; c < n; c += 32) {
      if (!resume) ub[c] = 0.0;
      s.u0s[c] = a.u0[(size_t)b * n + c];
    }
    if (!resume) {
#pragma unroll 1
      for (int e = lane; e < a.max_outer; e += 32) {
        a.cost_hist[(size_t)b * a.max_outer + e] = qnan;
        if (a.e_u_hist) a.e_u_hist[(size_t)b * a.max_outer + e] = qnan;
      }
    }
    if (lane < 2 * NJ) s.x0s[lane] = x0[lane];
    const double nrm0 = sqrt(warp_sum(part));
    const double cost0 = a.cost0[b];
    const double fupper = (a.has_bounds && a.fupper) ? a.fupper[b] : INFINITY;
    int status = -1, iters = 0, touched = 0, steps_prob = 0;
    if (resume) {
      iters = a.iters[b];
      touched = lane == 0 ? a.touch[b] : 0;
      steps_prob = a.prob_steps ? a.prob_steps[b] : 0;
    } else if (nrm0 < a.eps_outer) {
      status = 0;
    } else if (1 > a.max_outer) {
      status = 1;
    }
    __syncwarp();

    for (int it = iters + 1; status < 0; ++it) {
      // ---- get_con: distance + num_jac gradient of every waypoint, rows written in place (CFS_FANUC.m:110-124) ----
      if (PROF) pf_t1 = clock64();
#pragma unroll 1
      for (int i = lane; i < H; i += 32) {
        const double *thp = s.th + (size_t)i * NJ;
#pragma unroll 1
        for (int k = 0; k < NJ; ++k) {
          double sn, cs;
          sincos(thp[k] + tab.link[k].th_off, &sn, &cs);
          sc[(0 * NJ + k) * 32 + lane] = cs;
          sc[(1 * NJ + k) * 32 + lane] = sn;
        }
#pragma unroll 1
        for (int j0 = 0; j0 < O; j0 += OC) {
          double dist[OC];
          numjac_waypoint_lane<NJ, OC>(tab, sc, pm, lane, j0, O, touched, dist, s.ocoef, j0 * H + i, H);
#pragma unroll
          for (int jj = 0; jj < OC; ++jj) {
            if (j0 + jj >= O) continue;
            const int cid = (j0 + jj) * H + i;
            double margin = a.margin_is_D ? tab.obs[j0 + jj].D : tab.obs[j0 + jj].eps;
            if (OFF) margin = margin + a.margin_off[(size_t)b * OH + cid];
            double gu = 0.0, sg = 0.0;
#pragma unroll 1
            for (int k = 0; k < NJ; ++k) {
              const double gk = -s.ocoef[(size_t)cid * NJ + k];
              // s = I - Diff'*Bj*u (:120); B_theta u = theta_i - (theta_0 + i dt w_0) once x_ is the roll-out of u
              if (it > 1) gu += gk * (thp[k] - (s.x0s[k] + ((i + 1) * dt) * s.x0s[NJ + k]));
              const double gd = __ldg(a.gdiag + i * NJ + k);
              sg += (gk * gk) * (gd * gd);
            }
            s.orhs[cid] = (dist[jj] - margin) - gu;  // I = distance - margin (CFS_FANUC.m:117)
            s.onrm[cid] = sg;                        // scan normalisation (diagonal proxy of c QQ^-1 c')
          }
        }
      }
#pragma unroll 1
      for (int e = lane * 4; e < mz; e += 128)  // inact[] = 0, four rows per store (the region is padded to 16 B)
        *reinterpret_cast<unsigned int *>(s.inact + e) = 0u;
      __syncwarp();
      if (PROF) {
        const long long now = clock64();
        pf_grad += now - pf_t1;
        pf_t1 = now;
        ++pf_passes;
      }

      // ---- Solve_QP (CFS_FANUC.m:85) ----
      int q = 0, steps = 0;
      const int masked = w_mask_antiparallel<NJ>(s, P);
      const int qst = wqp_solve<NJ, LIM>(s, P, cost0, fupper, a.esc_steps, masked, q, steps, qmax_seen);
      if (PROF) pf_qp += clock64() - pf_t1;
      steps_total += steps;
      steps_prob += steps;
      if (qst != 0) {  // 2 infeasible / 3 numerical: u, x_ keep the previous iterate; 4: the heavy tier redoes this iteration
        status = qst;
        break;
      }
      // ---- e_u, cost by duality, roll-out, stop rule (EVAL.m:51-73, CFS_FANUC.m:88-94) ----
      double *dscr = s.zc;  // u_old - u_new: the direction cache is dead by now
      double cost = cost0;
      {
        double pc = 0.0;
#pragma unroll 1
        for (int w = 0; w < q; ++w) {
          const int cw = s.act[w];
          pc += s.lam[w] * (W_ROW_DOT(cw, s.u0s) - w_row_rhs<NJ, LIM>(cw, s, P));  // lambda_w * violation at u0
        }
        cost = cost0 + 0.5 * pc;
      }
      __syncwarp();
      double pe = 0.0;
#pragma unroll 2
      for (int c = lane; c < n; c += 32) {
        const double un = s.uq[c];
        const double uo = it > 1 ? ub[c] : 0.0;
        const double dlt = uo - un;
        pe += dlt * dlt;
        dscr[c] = dlt;
        ub[c] = un;
      }
      const double e_u = sqrt(warp_sum(pe));
      __syncwarp();
      // roll-out in closed form: theta_i = theta_0 + i dt w_0 + (B_theta u)_i, omega_i = w_0 + (B_omega u)_i (prefix sums);
      // ||x_new - x_old||: theta against the stored x_, omega against xref (first iteration) or through B_omega (u_old - u_new)
      double px = 0.0;
      {
        const int i0 = 2 * lane, i1 = i0 + 1;
        const bool v0 = i0 < H, v1 = i1 < H;
#pragma unroll 1
        for (int k = 0; k < NJ; ++k) {
          const double a0 = v0 ? s.uq[i0 * NJ + k] : 0.0, a1 = v1 ? s.uq[i1 * NJ + k] : 0.0;
          double s0, s1, t0, t1;
          w_prefix2(a0, a1, s0, s1, t0, t1);
          double dw0 = 0.0, dw1 = 0.0;  // omega_old - omega_new
          if (it > 1) {
            const double d0 = v0 ? dscr[i0 * NJ + k] : 0.0, d1 = v1 ? dscr[i1 * NJ + k] : 0.0;
            double r0, r1, q0, q1;
            w_prefix2(d0, d1, r0, r1, q0, q1);
            dw0 = dt * r0;
            dw1 = dt * r1;
          }
          const double w0 = s.x0s[NJ + k], th00 = s.x0s[k];
#pragma unroll 1
          for (int h = 0; h < 2; ++h) {
            if (!(h ? v1 : v0)) continue;
            const int i = h ? i1 : i0;
            const double S1 = h ? s1 : s0, T = h ? t1 : t0;
            const double thn = (th00 + ((i + 1) * dt) * w0) + dt2 * (0.5 * S1 + T), omn = w0 + dt * S1;
            double dw = h ? dw1 : dw0;
            if (it == 1) dw = xref[(size_t)i * 2 * NJ + NJ + k] - omn;
            const double dth = thn - s.th[i * NJ + k];
            px += dth * dth + dw * dw;
            s.th[i * NJ + k] = thn;
            xb[(size_t)i * 2 * NJ + k] = thn;
            xb[(size_t)i * 2 * NJ + NJ + k] = omn;
          }
        }
      }
      const double dx = sqrt(warp_sum(px));
      if (lane == 0) {
        a.cost_hist[(size_t)b * a.max_outer + (it - 1)] = cost;
        if (a.e_u_hist) a.e_u_hist[(size_t)b * a.max_outer + (it - 1)] = e_u;
      }
      iters = it;
      if (dx < a.eps_outer)
        status = 0;  // converged (EVAL.m:64-67)
      else if (it + 1 > a.max_outer)
        status = 1;  // MAX_ITER (EVAL.m:69-72)
      __syncwarp();
      if (a.it_stop && it >= a.it_stop) break;  // screening pass: the problem continues in a later launch
    }

    // ---- results: u and x_ of the last completed iteration are already in global memory ----
    if (PROF) pf_all += clock64() - pf_t0;
    const int any_touch = __any_sync(FULLMASK, touched);
    if (lane == 0) {
      a.iters[b] = iters;
      if (a.prob_steps) a.prob_steps[b] = steps_prob;
      if (status < 0) {  // screening pass: the problem continues in the next launch
        a.touch[b] = any_touch ? 0x100 : 0;
        a.cont_out[atomicAdd(a.cont_out_count, 1)] = b;
      } else {
        a.status[b] = status | (any_touch ? 0x100 : 0);
        if (status == 4) a.esc_list[atomicAdd(a.esc_count, 1)] = b;
      }
    }
  }
  if (lane == 0) {
    if (steps_total) atomicAdd(reinterpret_cast<unsigned long long *>(a.qp_steps), (unsigned long long)steps_total);
    if (qmax_seen) atomicMax(a.max_active, qmax_seen);
    if (PROF && a.prof) {  // slots 16..19 of the profile block: gradient-phase, QP, per-problem total cycles; gradient passes
      atomicAdd(reinterpret_cast<unsigned long long *>(a.prof + 16), (unsigned long long)pf_grad);
      atomicAdd(reinterpret_cast<unsigned long long *>(a.prof + 17), (unsigned long long)pf_qp);
      atomicAdd(reinterpret_cast<unsigned long long *>(a.prof + 18), (unsigned long long)pf_all);
      atomicAdd(reinterpret_cast<unsigned long long *>(a.prof + 19), (unsigned long long)pf_passes);
    }
  }
}

// ---- lock-step form: one outer iteration of the problems in list_cur, one warp per problem ------------------------------------
// The launch-per-iteration path (PSGCFS_FANUC.optimizer: the PSG point needs the batched QQ*u GEMM between two projections;
// DERIVEST gradients come from their own kernel) keeps its structure -- gradient kernel | QP kernel per outer iteration -- but
// the QP kernel (k_qp.cu: one CTA per problem) is replaced by this one: same prologue / epilogue, wqp_solve in the middle.
// Problems whose working set outgrows the warp tier are appended to esc_list and taken by k_qp in the same iteration.
template <int NJ, int NT, bool OFF = false, bool LIM = false>
__global__ void __launch_bounds__(NT, 3) k_qp_warp(SolveArgs a) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  constexpr int WPC = NT / 32;
  const int n = a.n, H = a.H, O = a.nobs, OH = O * H, m = OH + (LIM ? 6 : 4) * n, N = 2 * n;
  const int mz = LIM ? OH + 4 * n + (2 * n + 7) / 8 : m;  // bytes of the inact map (LIM: position rows as bits)
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const WarpSmem L = warp_smem(n, NJ, OH, a.warp_zs, WPC, 0, LIM);
  WView s = warp_view(smem_raw + L.regions + L.region_bytes * wid, n, NJ, OH, a.warp_zs);
  s.zgl = a.zslab + (size_t)(blockIdx.x * WPC + wid) * warp_slab_doubles(n, a.warp_zs);
  s.Mgl = s.zgl + (size_t)(WQ_QZ - a.warp_zs) * n;
  s.qcap = a.warp_qcap < WQ_QBIG - 1 ? (a.warp_qcap > 1 ? a.warp_qcap : 1) : WQ_QBIG - 1;
  const double dt = a.tab->dt, dt2 = dt * dt;
  const bool psg = a.solver == 1;
  const WDims P = {n, H, OH, O, m, 3 * n, a.has_lim, a.has_bounds, dt, a.G, a.gdiag, a.max_input, a.lim, LIM ? a.qlim : nullptr};
  const int count = *a.count_cur;
  const int it = a.outer_iter;
  long long steps_total = 0;
  int qmax_seen = 0;
  for (;;) {
    int slot = 0;
    if (lane == 0) slot = atomicAdd(a.work_counter, 1);
    slot = __shfl_sync(FULLMASK, slot, 0);
    if (slot >= count) break;
    const int b = a.list_cur[slot];
    const double *x0 = a.x0 + (size_t)b * 2 * NJ;
    double *ub = a.u + (size_t)b * n;
    double *xb = a.x + (size_t)b * N;
    __syncwarp();
    // ---- prologue: rows from the gradient kernel's output (CFS_FANUC.m:117-121), u0 ----
    if (lane < 2 * NJ) s.x0s[lane] = x0[lane];
#pragma unroll 2
    for (int c = lane; c < n; c += 32) s.u0s[c] = a.u0[(size_t)b * n + c];
#pragma unroll 1
    for (int e = lane * 4; e < mz; e += 128) *reinterpret_cast<unsigned int *>(s.inact + e) = 0u;
    __syncwarp();
#pragma unroll 1
    for (int cid = lane; cid < OH; cid += 32) {
      const int j = cid / H, i = cid - j * H;
      const double *gr = a.grad + ((size_t)b * OH + cid) * NJ;
      double margin = a.margin_is_D ? a.tab->obs[j].D : a.tab->obs[j].eps;
      if (OFF) margin = margin + a.margin_off[(size_t)b * OH + cid];
      double gu = 0.0, sg = 0.0;
#pragma unroll
      for (int k = 0; k < NJ; ++k) {
        const double gk = gr[k];
        s.ocoef[(size_t)cid * NJ + k] = -gk;
        // B_theta u = theta_i - (theta_0 + i dt w_0) once x_ is the roll-out of u (not in the first iteration: CFS_FANUC.m:55-56)
        if (it > 1) gu += gk * (xb[(size_t)i * 2 * NJ + k] - (s.x0s[k] + ((i + 1) * dt) * s.x0s[NJ + k]));
        const double gd = __ldg(a.gdiag + i * NJ + k);
        sg += (gk * gk) * (gd * gd);
      }
      s.orhs[cid] = (a.dist[(size_t)b * OH + cid] - margin) - gu;
      s.onrm[cid] = sg;
    }
    __syncwarp();
    // ---- the QP (CFS_FANUC.m:85) / the projection (PSGCFS_FANUC.m:120) ----
    int q = 0, steps = 0, status = 0;
    const bool skip_solve = psg && a.skip[b];  // stop_inner() already true: u stays, no projection (PSGCFS_FANUC.m:88)
    if (skip_solve) {
#pragma unroll 2
      for (int c = lane; c < n; c += 32) s.uq[c] = ub[c];
      __syncwarp();
    } else {
      const int masked = w_mask_antiparallel<NJ>(s, P);
      status = wqp_solve<NJ, LIM>(s, P, a.cost0[b], (a.has_bounds && a.fupper) ? a.fupper[b] : INFINITY, 0x7fffffff, masked, q, steps,
                             qmax_seen);
    }
    steps_total += steps;
    if (status == 4) {  // the working set outgrew the warp tier: k_qp redoes this problem's iteration
      if (lane == 0) a.esc_list[atomicAdd(a.esc_count, 1)] = b;
      continue;
    }
    if (lane == 0 && a.prob_steps) a.prob_steps[b] += steps;
    if (status != 0) {  // 2 infeasible / 3 numerical: u, x keep the previous iterate
      if (lane == 0) a.status[b] = status;
      continue;
    }
    // ---- epilogue: e_u, cost by duality, roll-out, stop rule (EVAL.m:51-73, CFS_FANUC.m:88-94) ----
    double cost = 0.0;
    if (!psg) {
      double pc = 0.0;
#pragma unroll 1
      for (int w = 0; w < q; ++w) {
        const int cw = s.act[w];
        pc += s.lam[w] * (W_ROW_DOT(cw, s.u0s) - w_row_rhs<NJ, LIM>(cw, s, P));
      }
      cost = a.cost0[b] + 0.5 * pc;
    }
    double pe = 0.0;
#pragma unroll 2
    for (int c = lane; c < n; c += 32) {
      const double un = s.uq[c];
      const double dlt = ub[c] - un;
      pe += dlt * dlt;
      ub[c] = un;
    }
    const double e_u = sqrt(warp_sum(pe));
    double px = 0.0;
    {
      const int i0 = 2 * lane, i1 = i0 + 1;
      const bool v0 = i0 < H, v1 = i1 < H;
#pragma unroll 1
      for (int k = 0; k < NJ; ++k) {
        const double a0 = v0 ? s.uq[i0 * NJ + k] : 0.0, a1 = v1 ? s.uq[i1 * NJ + k] : 0.0;
        double s0, s1, t0, t1;
        w_prefix2(a0, a1, s0, s1, t0, t1);
        const double w0 = s.x0s[NJ + k], th00 = s.x0s[k];
#pragma unroll 1
        for (int h = 0; h < 2; ++h) {
          if (!(h ? v1 : v0)) continue;
          const int i = h ? i1 : i0;
          const double S1 = h ? s1 : s0, T = h ? t1 : t0;
          const double thn = (th00 + ((i + 1) * dt) * w0) + dt2 * (0.5 * S1 + T), omn = w0 + dt * S1;
          // CFS: x_old = previous x_ (CFS_FANUC.m:88); PSGCFS never updates eval.x_old, it stays ones (EVAL.m:47)
          const double d1 = thn - (psg ? 1.0 : xb[(size_t)i * 2 * NJ + k]), d2 = omn - (psg ? 1.0 : xb[(size_t)i * 2 * NJ + NJ + k]);
          px += d1 * d1 + d2 * d2;
          xb[(size_t)i * 2 * NJ + k] = thn;
          xb[(size_t)i * 2 * NJ + NJ + k] = omn;
        }
      }
    }
    const double dx = sqrt(warp_sum(px));
    if (lane == 0) {
      if (!psg) a.cost_hist[(size_t)b * a.max_outer + (it - 1)] = cost;
      if (a.e_u_hist) a.e_u_hist[(size_t)b * a.max_outer + (it - 1)] = e_u;
      a.iters[b] = it;
      if (dx < a.eps_outer)
        a.status[b] = 0;
      else if (it + 1 > a.max_outer)
        a.status[b] = 1;
      else
        a.list_next[atomicAdd(a.count_next, 1)] = b;
    }
  }
  if (lane == 0) {
    if (steps_total) atomicAdd(reinterpret_cast<unsigned long long *>(a.qp_steps), (unsigned long long)steps_total);
    if (qmax_seen) atomicMax(a.max_active, qmax_seen);
  }
}

// ---- host side ------------------------------------------------------------------------------------------------------------
// CTA shapes (warps of one CTA share nothing but the staged tables; small CTAs let another context's launch move into an SM
// as soon as a few warps have drained):  cfg 0: 12 warps x 1 CTA/SM, 1: 3 warps x 3, 2: 4 warps x 3, 3: 1 warp x 10, 4: 2 warps x 5
#define WARP_NCFG 5
static const int kWarpNT[WARP_NCFG] = {384, 96, 128, 32, 64};

size_t warp_smem_bytes(const SolveArgs &a, int cfg) {
  return warp_smem(a.n, a.nj, a.nobs * a.H, a.warp_zs, kWarpNT[cfg] / 32, a.nobs, a.qlim != nullptr).total;
}

bool warp_supported(const SolveArgs &a, int cfg) {
  if (cfg < 0 || cfg >= WARP_NCFG) return false;
  if (a.nj != 2 && a.nj != 5) return false;
  if (a.H > 64 || a.n > 32 * W_NC) return false;  // two waypoints per lane in the prefix sums; W_NC controls per lane
  if (a.warp_zs < 1 || a.warp_zs > 8) return false;
  return warp_smem_bytes(a, cfg) <= 227 * 1024;
}

int warp_warps_per_cta(int cfg) { return kWarpNT[cfg] / 32; }
size_t warp_slab_bytes_per_warp(const SolveArgs &a) { return sizeof(double) * warp_slab_doubles(a.n, a.warp_zs); }

typedef void (*WarpKernel)(SolveArgs);
template <int NJ, bool OFF, bool LIM = false>
static WarpKernel warp_kernel_nj(int cfg, bool two) {
  switch (cfg) {
    case 0: return two ? k_cfs_warp<NJ, 384, 168, 2, false, OFF, LIM> : k_cfs_warp<NJ, 384, 168, 1, false, OFF, LIM>;
    case 1: return two ? k_cfs_warp<NJ, 96, 224, 2, false, OFF, LIM> : k_cfs_warp<NJ, 96, 224, 1, false, OFF, LIM>;
    case 2: return two ? k_cfs_warp<NJ, 128, 168, 2, false, OFF, LIM> : k_cfs_warp<NJ, 128, 168, 1, false, OFF, LIM>;
    case 3: return two ? k_cfs_warp<NJ, 32, 168, 2, false, OFF, LIM> : k_cfs_warp<NJ, 32, 168, 1, false, OFF, LIM>;
    case 4: return two ? k_cfs_warp<NJ, 64, 168, 2, false, OFF, LIM> : k_cfs_warp<NJ, 64, 168, 1, false, OFF, LIM>;
  }
  return nullptr;
}
// off: the margin-offset instantiations (a.margin_off != nullptr); lim: the joint-limit ones (a.qlim != nullptr, always with
// offsets).  The phase profile has neither (timing level 3 measures the unchecked solve).
static WarpKernel warp_kernel(int nj, int cfg, int nobs, bool prof = false, bool off = false, bool lim = false) {
  if (prof && !off && nj == 5 && cfg == 3 && nobs <= 1) return k_cfs_warp<5, 32, 168, 1, true>;
  if (lim && !off) return nullptr;
  if (nj == 2)
    return lim ? warp_kernel_nj<2, true, true>(cfg, nobs > 1)
               : (off ? warp_kernel_nj<2, true>(cfg, nobs > 1) : warp_kernel_nj<2, false>(cfg, nobs > 1));
  if (nj == 5)
    return lim ? warp_kernel_nj<5, true, true>(cfg, nobs > 1)
               : (off ? warp_kernel_nj<5, true>(cfg, nobs > 1) : warp_kernel_nj<5, false>(cfg, nobs > 1));
  return nullptr;
}

int warp_max_grid(const SolveArgs &a, int device, int cfg) {
  const size_t smem = warp_smem_bytes(a, cfg);
  WarpKernel k = warp_kernel(a.nj, cfg, a.nobs, false, a.margin_off != nullptr, a.qlim != nullptr);
  if (!k) return 0;
  int sms = 0, per = 0;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
  // the opt-in maximum, not this configuration's size: the attribute is per function and shared by every context of the process
  if (smem > 227 * 1024 || cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) != cudaSuccess) return 0;
  // all of the SM's 228 KB as shared memory: the resident CTAs are limited by their shared-memory regions, not by L1
  cudaFuncSetAttribute(k, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per, k, kWarpNT[cfg], smem);
  return sms * per;
}

cudaError_t launch_warp(const SolveArgs &a, int grid, int cfg, cudaStream_t st) {
  const bool off = a.margin_off != nullptr;
  WarpKernel k = warp_kernel(a.nj, cfg, a.nobs, a.prof != nullptr, off, a.qlim != nullptr);
  if (!k) return cudaErrorInvalidValue;
  if (a.prof && !off) {  // the profiled instantiation is a function of its own: same opt-in limits as warp_max_grid sets
    cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    cudaFuncSetAttribute(k, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  }
  k<<<grid, kWarpNT[cfg], warp_smem_bytes(a, cfg), st>>>(a);
  return cudaGetLastError();
}

// lock-step warp QP (PSGCFS / DERIVEST paths): 4 warps per CTA
bool qp_warp_supported(const SolveArgs &a) {
  if (a.nj != 2 && a.nj != 5) return false;
  if (a.H > 64 || a.n > 32 * W_NC || a.warp_zs < 1 || a.warp_zs > 8) return false;
  return warp_smem(a.n, a.nj, a.nobs * a.H, a.warp_zs, 4, 0, a.qlim != nullptr).total <= 227 * 1024;
}

static WarpKernel qp_warp_kernel(const SolveArgs &a) {
  const bool off = a.margin_off != nullptr, lim = a.qlim != nullptr;
  if (lim && !off) return nullptr;
  if (a.nj == 2) return lim ? k_qp_warp<2, 128, true, true> : (off ? k_qp_warp<2, 128, true> : k_qp_warp<2, 128>);
  if (a.nj == 5) return lim ? k_qp_warp<5, 128, true, true> : (off ? k_qp_warp<5, 128, true> : k_qp_warp<5, 128>);
  return nullptr;
}

int qp_warp_max_grid(const SolveArgs &a, int device) {
  const size_t smem = warp_smem(a.n, a.nj, a.nobs * a.H, a.warp_zs, 4, 0, a.qlim != nullptr).total;
  WarpKernel k = qp_warp_kernel(a);
  if (!k) return 0;
  int sms = 0, per = 0;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
  if (cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) != cudaSuccess) return 0;
  cudaFuncSetAttribute(k, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per, k, 128, smem);
  return sms * per;
}

cudaError_t launch_qp_warp(const SolveArgs &a, int grid, cudaStream_t st) {
  const size_t smem = warp_smem(a.n, a.nj, a.nobs * a.H, a.warp_zs, 4, 0, a.qlim != nullptr).total;
  WarpKernel k = qp_warp_kernel(a);
  if (!k) return cudaErrorInvalidValue;
  k<<<grid, 128, smem, st>>>(a);
  return cudaGetLastError();
}

}  // namespace cfs
