// k_qp.cu -- K2+K3+K4: constraint assembly, batched strictly-convex QP, roll-out, cost and stop rule (sm_100a).
//
// Replaces, per outer iteration and per problem (reference file:line):
//   Lib/CFS_FANUC.m:119-129   get_con row assembly  (l=-Diff'*Bj(1:njoint,:), s=I-Diff'*Bj*u, velocity rows)
//   Lib/CFS_FANUC.m:85        quadprog(QQ,ff,Ainq,binq,[],[],-MAX_input,MAX_input)
//   Lib/PSGCFS_FANUC.m:120    quadprog(I,-u_,Ainq,binq)                       (projection, identity metric)
//   Lib/CFS_FANUC.m:90-94     roll-out xR(:,i)=A*xR(:,i-1)+B*u_i
//   Lib/EVAL.m:51-73          get_cost, store_result, stop_outer
//
// Design (B200-first, not a translation of quadprog):
//   * persistent CTAs pull problems from a device work queue (no host round trip, no tail of idle SMs);
//   * the QP is solved by a dual active-set method (Goldfarb-Idnani) written entirely in "primitive space":
//     v = P u (3n values: joint displacements B_theta u, joint velocities B_omega u, controls u) lives in shared
//     memory; every constraint reads <= nj entries of v, and every metric inner product the method needs is a small
//     bilinear form over the batch-shared Gram matrix G = P QQ^{-1} P' (k_setup.cu) held in L2.  No n x n
//     per-problem factorisation, no dense Ainq (550 x 250 per problem in the reference) is ever formed;
//   * the only per-problem matrix is the inverse of the working-set Gram matrix (q x q, q = #active rows, typically
//     < 8): in shared memory up to q = QP_QS, spilled to a per-CTA global slab beyond, rank-1 updated on add / drop;
//   * the primal point is never stepped: at the top of every outer step v is re-evaluated from the multipliers,
//     v = v0 - G (C_W' lambda), as one pass over the flat list of active (primitive row, weight) terms with many
//     independent L2 loads in flight (small working sets: all 3n entries straight from G; large ones: the n control
//     entries from G followed by the closed-form B_theta / B_omega sums).  The inner loop only needs scalars;
//   * the optimal cost comes from duality: f(u) = f(u0) + 1/2 sum_w lambda_w * (violation of row w at u0).
#include "qp_core.cuh"

namespace cfs {

size_t qp_smem_bytes(const SolveArgs &a) {
  size_t off[QP_NOFF];
  const int OH = a.nobs * a.H;
  const bool lim = a.qlim != nullptr;
  return qp_smem_layout(a.n, a.nj, OH, OH + (lim ? 6 : 4) * a.n, off, QP_QS, QP_THREADS, 0, lim);
}


// ============================================================================================================
// The kernel
// ============================================================================================================
// OFF: the obstacle rows read a.margin_off (per-waypoint margin offsets of the checked solve); a separate instantiation, the one
// without it is unchanged.  LIM (only with OFF): the QP also has the joint position rows of a.qlim.
template <bool OFF, bool LIM = false>
__global__ void __launch_bounds__(QP_THREADS, 3) k_qp(SolveArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int n = a.n, nj = a.nj, H = a.H, np = 3 * n, OH = a.nobs * H, m = OH + (LIM ? 6 : 4) * n;
  const int tid = threadIdx.x;
  const QpView s = qp_view(smem_raw, n, nj, OH, m, QP_QS, QP_THREADS, 0, LIM);
  const double *__restrict__ G = a.G;
  const double *__restrict__ gnorm = a.gdiag;  // sqrt(diag(G))
  const int has_vel = a.has_lim, has_bnd = a.has_bounds;
  const bool psg = a.solver == 1;
  for (int e = tid; e < 3 * n; e += QP_THREADS) s.gns[e] = gnorm[e] * gnorm[e];  // G_ii
  for (int e = tid; e < n; e += QP_THREADS) s.ums[e] = has_bnd ? a.max_input[e] : 0.0;
  const double *umax = s.ums;
  const double dt = a.tab->dt;
  const int ldg = a.slab_ld;
  double *Mgl = a.slab + (size_t)blockIdx.x * ldg * ldg;  // spill area of the working-set inverse
  const int count = *a.count_cur;
  long long steps_total = 0;
  int qmax_seen = 0;
  // optional phase profile (thread 0 clocks): 0 prologue, 1 refresh, 2 scan, 3 gram+solve+steplen, 4 update, 5 epilogue,
  // 6 problems, 7 outer steps
  long long pf[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  long long tck = 0;
  const bool prof = a.prof != nullptr;
  const QpDims dims = {n, nj, H, np, OH, m, has_vel, has_bnd, G, umax, Mgl, ldg, dt};

  for (;;) {
    __syncthreads();
    if (tid == 0) s.ctl[0] = atomicAdd(a.work_counter, 1);
    __syncthreads();
    const int slot = s.ctl[0];
    if (slot >= count) break;
    const int b = a.list_cur[slot];
    const double *x0 = a.x0 + (size_t)b * 2 * nj;
    double *ub = a.u + (size_t)b * n;
    double *xb = a.x + (size_t)b * 2 * n;
    const double *v0 = a.v0 + (size_t)b * np;

    // ---- prologue: v = v0; disp = B_theta u_cur; obstacle rows ------------------------------------------------
    PF_START();
    for (int pi = tid; pi < np; pi += QP_THREADS) {
      const double t_ = v0[pi];
      s.v0s[pi] = t_;
      s.v[pi] = t_;
    }
    for (int e = tid; e < m; e += QP_THREADS) s.inact[e] = 0;
    if (tid < 8) {
      s.lim[tid] = (tid < nj && has_vel) ? a.lim[tid] : 0.0;
      s.w0[tid] = (tid < nj) ? x0[nj + tid] : 0.0;
      if (LIM) {  // qmax | qmin | theta0 of the joint position rows
        s.lim[8 + tid] = (tid < nj) ? a.qlim[tid] : 0.0;
        s.lim[16 + tid] = (tid < nj) ? a.qlim[nj + tid] : 0.0;
        s.lim[24 + tid] = (tid < nj) ? x0[tid] : 0.0;
      }
    }
    // disp(i,k) = (Bj(1:njoint,:)*u)(k) of CFS_FANUC.m:120 -> s.g.  In the first outer iteration u = 0 (CFS_FANUC.m:56)
    // while x_ is the reference line; afterwards x_ is the roll-out of u, so B_theta u = theta_i - (theta_0 + i dt w_0).
    for (int e = tid; e < n; e += QP_THREADS) {
      const int i = e / nj, k = e % nj;
      s.g[e] = (a.outer_iter == 1) ? 0.0 : xb[(size_t)i * 2 * nj + k] - (x0[k] + ((i + 1) * dt) * x0[nj + k]);
    }
    __syncthreads();
    for (int cid = tid; cid < OH; cid += QP_THREADS) {
      const int j = cid / H, i = cid % H;
      const double *gr = a.grad + ((size_t)b * OH + cid) * nj;
      const double dist = a.dist[(size_t)b * OH + cid];
      double margin = a.margin_is_D ? a.tab->obs[j].D : a.tab->obs[j].eps;
      if (OFF) margin = margin + a.margin_off[(size_t)b * OH + cid];
      double gu = 0.0;
      for (int k = 0; k < nj; ++k) {
        s.ocoef[cid * nj + k] = -gr[k];                 // l = -Diff'*Bj(1:njoint,:)   (CFS_FANUC.m:121)
        gu += gr[k] * s.g[i * nj + k];
      }
      s.orhs[cid] = (dist - margin) - gu;               // s = I - Diff'*Bj*u          (CFS_FANUC.m:117,120)
    }
    __syncthreads();
    for (int cid = tid; cid < OH; cid += QP_THREADS) {
      const int i = cid % H;
      double sg = 0.0;
      for (int k = 0; k < nj; ++k) sg += s.ocoef[cid * nj + k] * s.ocoef[cid * nj + k] * s.gns[i * nj + k];
      s.onrm[cid] = sg;  // scan normalisation (diagonal proxy of c QQ^-1 c')
    }
    if (tid == 0) s.toff[0] = 0;
    __syncthreads();
    PF_ADD(0);
    pf[6] += 1;

    // ---- dual active-set iterations --------------------------------------------------------------------------
    int q = 0, steps = 0;
    const bool skip_solve = psg && a.skip[b];
    if (skip_solve) {  // stop_inner() already true: u stays, no projection (PSGCFS_FANUC.m:88)
      for (int c = tid; c < n; c += QP_THREADS) s.v[2 * n + c] = ub[c];
      __syncthreads();
    }
    const int masked = skip_solve ? 0 : qp_mask_antiparallel<QP_THREADS>(s, dims);
    double fup = (has_bnd && a.fupper) ? a.fupper[b] : INFINITY;
    if (psg && has_vel && !skip_solve) {
      // Weak-duality bound for the projection (PSGCFS_FANUC.m:115-128 has no control bounds): the velocity rows alone confine
      // every feasible u to |u_(i,k)| <= max(2 lim_k, lim_k + |w0_k|) / dt =: U_k (two consecutive velocities inside
      // [-lim, lim]), so 1/2 ||u - u_||^2 <= 1/2 sum (U_k + |u__(i,k)|)^2 on the feasible set.  A dual value above it proves
      // infeasibility -- long before the nearly dependent working set of an infeasible projection ruins the inverse.
      double part = 0.0;
      for (int c = tid; c < n; c += QP_THREADS) {
        const int k = c % nj;
        const double U = fmax(2.0 * s.lim[k], s.lim[k] + fabs(s.w0[k])) / dt + fabs(s.v0s[2 * n + c]);
        part += U * U;
      }
      fup = a.cost0[b] + 0.5 * block_sum<QP_THREADS>(part, s.red) * (1.0 + 1e-9);
    }
    const int status = qp_solve<QP_THREADS, QP_QS, true, 0, 0, LIM>(s, dims, a.cost0[b], fup, skip_solve, q, steps,
                                qmax_seen, pf, tck, prof, 0x7fffffff, masked);
    steps_total += steps;
    if (tid == 0 && a.prob_steps) a.prob_steps[b] += steps;

    // ---- epilogue ------------------------------------------------------------------------------------------------
    const int it = a.outer_iter;  // 1-based
    if (status == 0) {
      // u = control block of v; e_u = ||u_old - u||   (EVAL.m:58)
      double pe = 0.0;
      for (int c = tid; c < n; c += QP_THREADS) {
        const double un = s.v[2 * n + c];
        const double dlt = ub[c] - un;
        pe += dlt * dlt;
        ub[c] = un;
      }
      const double e_u = sqrt(block_sum<QP_THREADS>(pe, s.red));
      // cost by duality: f(u) = f(u0) + 1/2 sum_w lam_w * (c_w u0 - rhs_w)
      double pc = 0.0;
      for (int w = tid; w < q; w += QP_THREADS) {
        const double val0 = -slack_at<0, LIM>(s.act[w], dims, s, s.v0s);
        pc += s.lam[w] * val0;
      }
      const double cost = psg ? 0.0 : a.cost0[b] + 0.5 * block_sum<QP_THREADS>(pc, s.red);  // PSGCFS: k_psg_cost
      // roll-out (CFS_FANUC.m:90-94): x_old is staged in shared memory (coalesced), nj threads run the recurrence
      // xR(:,i) = A xR(:,i-1) + B u_i there, then the new trajectory is written back coalesced; ||x_new - x_old||^2
      // (EVAL.m:64) is accumulated on the way.  xbuf aliases the term-weight scratch (tcoef|twgt), free by now.
      double *xbuf = s.tcoef;
      __syncthreads();
      for (int e = tid; e < 2 * n; e += QP_THREADS) xbuf[e] = xb[e];
      __syncthreads();
      double px = 0.0;
      if (tid < nj) {
        double th = x0[tid], om = x0[nj + tid];
        for (int i = 0; i < H; ++i) {
          const double uk = s.v[2 * n + i * nj + tid];
          const double thn = (th + dt * om) + (0.5 * dt * dt) * uk;
          const double omn = om + dt * uk;
          th = thn;
          om = omn;
          double *xs = xbuf + (size_t)i * 2 * nj;
          // CFS: x_old = previous x_ (CFS_FANUC.m:88); PSGCFS never updates eval.x_old, it stays ones (EVAL.m:47)
          const double d1 = th - (psg ? 1.0 : xs[tid]), d2 = om - (psg ? 1.0 : xs[nj + tid]);
          px += d1 * d1 + d2 * d2;
          xs[tid] = th;
          xs[nj + tid] = om;
        }
      }
      __syncthreads();
      for (int e = tid; e < 2 * n; e += QP_THREADS) xb[e] = xbuf[e];
      const double dx = sqrt(block_sum<QP_THREADS>(px, s.red));
      if (tid == 0) {
        if (!psg) a.cost_hist[(size_t)b * a.max_outer + (it - 1)] = cost;
        if (a.e_u_hist) a.e_u_hist[(size_t)b * a.max_outer + (it - 1)] = e_u;
        a.iters[b] = it;
        if (dx < a.eps_outer) {
          a.status[b] = 0;  // converged (EVAL.m:64-67)
        } else if (it + 1 > a.max_outer) {
          a.status[b] = 1;  // MAX_ITER (EVAL.m:69-72)
        } else {
          a.list_next[atomicAdd(a.count_next, 1)] = b;
        }
      }
    } else if (tid == 0) {
      a.status[b] = status;  // 2 infeasible / 3 numerical: u, x keep the previous iterate
    }
    PF_ADD(5);
  }
  if (a.prof && tid == 0)
    for (int k = 0; k < 8; ++k)
      if (pf[k]) atomicAdd(reinterpret_cast<unsigned long long *>(a.prof + k), (unsigned long long)pf[k]);
  if (tid == 0) {
    if (steps_total) atomicAdd(reinterpret_cast<unsigned long long *>(a.qp_steps), (unsigned long long)steps_total);
    if (qmax_seen) atomicMax(a.max_active, qmax_seen);
  }
}

// the margin-offset instantiation when a.margin_off is set, the joint-limit one (which also reads the offsets) when a.qlim is set
static void (*qp_kernel(const SolveArgs &a))(SolveArgs) {
  if (a.qlim) return a.margin_off ? k_qp<true, true> : nullptr;
  return a.margin_off ? k_qp<true> : k_qp<false>;
}

int qp_max_grid(const SolveArgs &a, int device) {
  int sms = 0, per = 0;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
  const size_t smem = qp_smem_bytes(a);
  void (*k)(SolveArgs) = qp_kernel(a);
  if (!k) return 0;
  cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per, k, QP_THREADS, smem);
  if (per < 1) per = 1;
  return sms * per;
}

cudaError_t launch_qp(const SolveArgs &a, int grid, cudaStream_t st) {
  const size_t smem = qp_smem_bytes(a);
  void (*k)(SolveArgs) = qp_kernel(a);
  if (!k) return cudaErrorInvalidValue;
  k<<<grid, QP_THREADS, smem, st>>>(a);
  return cudaGetLastError();
}

// ============================================================================================================
// Batch initialisation
// ============================================================================================================
// one CTA per problem: u=0, x_=sys_info.x_ (CFS_FANUC.m:55-56), histories NaN, first stop_outer test with
// x_old = ones (EVAL.m:47,61-73), initial active list.
__global__ void __launch_bounds__(128) k_solve_init(SolveArgs a) {
  __shared__ double red[(QP_THREADS / 32)];
  const int b = blockIdx.x, tid = threadIdx.x;
  const int n = a.n, N = 2 * n;
  double part = 0.0;
  for (int e = tid; e < N; e += blockDim.x) {
    const double xv = a.xref[(size_t)b * N + e];
    a.x[(size_t)b * N + e] = xv;
    part += (xv - 1.0) * (xv - 1.0);
  }
  for (int e = tid; e < n; e += blockDim.x) a.u[(size_t)b * n + e] = 0.0;
  for (int e = tid; e < a.max_outer; e += blockDim.x) {
    a.cost_hist[(size_t)b * a.max_outer + e] = __longlong_as_double(0x7ff8000000000000LL);
    if (a.e_u_hist) a.e_u_hist[(size_t)b * a.max_outer + e] = __longlong_as_double(0x7ff8000000000000LL);
  }
  const double nrm = sqrt(block_sum<QP_THREADS>(part, red));
  if (tid == 0) {
    a.iters[b] = 0;
    a.flags[b] = 0;
    if (a.solver == 1) {
      a.cost_old[b] = 100000.0;   // EVAL.m:29
      a.cost_new[b] = a.caug[b];  // get_cost(u = 0), PSGCFS_FANUC.m:66
      a.skip[b] = 0;
    }
    if (nrm < a.eps_outer) {
      a.status[b] = 0;
    } else if (1 > a.max_outer) {
      a.status[b] = 1;
    } else {
      a.status[b] = -1;
      a.list_cur[atomicAdd(a.count_cur, 1)] = b;
    }
  }
}

cudaError_t launch_solve_init(const SolveArgs &a, cudaStream_t s) {
  if (a.B <= 0) return cudaSuccess;
  k_solve_init<<<a.B, 128, 0, s>>>(a);
  return cudaGetLastError();
}

// v0 = P u0 and cost0 = caug + 1/2 ff'u0 (value of EVAL.get_cost at the unconstrained minimiser), one CTA per problem
__global__ void __launch_bounds__(128) k_v0(SolveArgs a) {
  __shared__ double red[(QP_THREADS / 32)];
  extern __shared__ double u0s[];
  const int b = blockIdx.x, tid = threadIdx.x;
  const int n = a.n, nj = a.nj, np = 3 * n;
  const double dt = a.tab->dt;
  double part = 0.0;
  for (int e = tid; e < n; e += blockDim.x) {
    const double uv = a.u0[(size_t)b * n + e];
    u0s[e] = uv;
    part += a.ff[(size_t)b * n + e] * uv;
  }
  const double fu = block_sum<QP_THREADS>(part, red);
  if (tid == 0) a.cost0[b] = a.caug[b] + 0.5 * fu;
  if (a.fupper) {  // sup over the box |u|<=MAX_input of EVAL.get_cost: 1/2 ||QQ||_inf sum umax^2 + sum |ff| umax + caug
    double pb = 0.0;
    if (a.has_bounds)
      for (int e = tid; e < n; e += blockDim.x) {
        const double um = a.max_input[e];
        pb += 0.5 * a.qq_norm_inf * um * um + fabs(a.ff[(size_t)b * n + e]) * um;
      }
    const double sb = block_sum<QP_THREADS>(pb, red);
    if (tid == 0) a.fupper[b] = a.has_bounds ? (fabs(a.caug[b]) + sb) * (1.0 + 1e-6) + 1e-6 : INFINITY;
  }
  for (int pi = tid; pi < np; pi += blockDim.x) {
    double acc;
    if (pi < n) {
      const int i = pi / nj, k = pi % nj;
      acc = 0.0;
      for (int j = 0; j <= i; ++j) acc += (0.5 * dt * dt + ((i - j) * dt) * dt) * u0s[j * nj + k];
    } else if (pi < 2 * n) {
      const int qq = pi - n, i = qq / nj, k = qq % nj;
      acc = 0.0;
      for (int j = 0; j <= i; ++j) acc += dt * u0s[j * nj + k];
    } else {
      acc = u0s[pi - 2 * n];
    }
    a.v0[(size_t)b * np + pi] = acc;
  }
}

cudaError_t launch_v0(const SolveArgs &a, cudaStream_t s) {
  if (a.B <= 0) return cudaSuccess;
  k_v0<<<a.B, 128, sizeof(double) * a.n, s>>>(a);
  return cudaGetLastError();
}

// problems still marked running (-1) after the last launched iteration cannot exist; flags are merged into status here
__global__ void k_finalize(SolveArgs a) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= a.B) return;
  int st = a.status[b];
  if (st < 0) st = 1;
  a.status[b] = st | (a.flags[b] & 0x100);
}

cudaError_t launch_finalize(const SolveArgs &a, cudaStream_t s) {
  if (a.B <= 0) return cudaSuccess;
  k_finalize<<<(a.B + 127) / 128, 128, 0, s>>>(a);
  return cudaGetLastError();
}

// ---- K5: PSG_update_arm (PSGCFS_FANUC.m:106-112), one CTA per active problem ------------------------------------
//   u_ = u - alpha*((QQ*u + ff) + 10*noise/(iter_O^2+1));   then v0 = P u_ for the projection QP (Hessian I, no bounds).
// stop_inner (PSGCFS_FANUC.m:136-142) is evaluated first: |cost_new - cost_old| < epsilon_I = 1e-4 skips the step.
__global__ void __launch_bounds__(128) k_psg_point(SolveArgs a) {
  extern __shared__ double u0s[];
  if ((int)blockIdx.x >= *a.count_cur) return;
  const int b = a.list_cur[blockIdx.x], tid = threadIdx.x;
  const int n = a.n, nj = a.nj, np = 3 * n;
  const double dt = a.tab->dt;
  const double cn = a.cost_new[b], co = a.cost_old[b];
  if (fabs(cn - co) < 1e-4) {  // uniform across the CTA
    if (tid == 0) a.skip[b] = 1;
    return;
  }
  const double it = (double)a.outer_iter;
  const double *nz = a.noise ? a.noise + ((size_t)b * a.max_outer + (a.outer_iter - 1)) * n : nullptr;
  for (int e = tid; e < n; e += blockDim.x) {
    const double g = a.w[(size_t)b * n + e] + a.ff[(size_t)b * n + e];
    const double uv = a.u[(size_t)b * n + e] - a.alpha * (g + 10 * (nz ? nz[e] : 0.0) / (it * it + 1));
    u0s[e] = uv;
    a.u0[(size_t)b * n + e] = uv;
  }
  if (tid == 0) {
    a.skip[b] = 0;
    a.cost_old[b] = cn;  // PSGCFS_FANUC.m:89
    a.cost0[b] = 0.0;
  }
  __syncthreads();
  for (int pi = tid; pi < np; pi += blockDim.x) {
    double acc;
    if (pi < n) {
      const int i = pi / nj, k = pi % nj;
      acc = 0.0;
      for (int j = 0; j <= i; ++j) acc += (0.5 * dt * dt + ((i - j) * dt) * dt) * u0s[j * nj + k];
    } else if (pi < 2 * n) {
      const int qq = pi - n, i = qq / nj, k = qq % nj;
      acc = 0.0;
      for (int j = 0; j <= i; ++j) acc += dt * u0s[j * nj + k];
    } else {
      acc = u0s[pi - 2 * n];
    }
    a.v0[(size_t)b * np + pi] = acc;
  }
}

cudaError_t launch_psg_point(const SolveArgs &a, cudaStream_t s) {
  if (a.B <= 0) return cudaSuccess;
  k_psg_point<<<a.B, 128, sizeof(double) * a.n, s>>>(a);
  return cudaGetLastError();
}

// EVAL.get_cost (EVAL.m:51-53) of the projected iterate, w = QQ*u from the batched GEMM; one CTA per problem of the list
// the QP kernel just consumed.  Problems whose projection failed this iteration (iters[b] != outer_iter) are skipped.
__global__ void __launch_bounds__(128) k_psg_cost(SolveArgs a) {
  __shared__ double red[(QP_THREADS / 32)];
  if ((int)blockIdx.x >= *a.count_cur) return;
  const int b = a.list_cur[blockIdx.x], tid = threadIdx.x, n = a.n;
  if (a.iters[b] != a.outer_iter) return;
  double pq = 0.0, pl = 0.0;
  for (int e = tid; e < n; e += blockDim.x) {
    const double uv = a.u[(size_t)b * n + e];
    pq += uv * a.w[(size_t)b * n + e];
    pl += uv * a.ff[(size_t)b * n + e];
  }
  const double quad = block_sum<QP_THREADS>(pq, red);
  const double lin = block_sum<QP_THREADS>(pl, red);
  if (tid == 0) {
    const double cost = (0.5 * quad + lin) + a.caug[b];
    a.cost_new[b] = cost;
    a.cost_hist[(size_t)b * a.max_outer + (a.outer_iter - 1)] = cost;
  }
}

cudaError_t launch_psg_cost(const SolveArgs &a, cudaStream_t s) {
  if (a.B <= 0) return cudaSuccess;
  k_psg_cost<<<a.B, 128, 0, s>>>(a);
  return cudaGetLastError();
}

// ============================================================================================================
// Dense get_con rows for one problem, in the reference's order (CFS_FANUC.m:110-131); parity/debug entry.
// ============================================================================================================
__global__ void k_get_con_rows(const DevTables *tab, int H, int nj, int nobs, int has_lim, int margin_is_D,
                               const double *x0, const double *u, const double *lim, const double *dist,
                               const double *grad, double *Ainq, double *binq, int m) {
  const int n = H * nj;
  const int per = has_lim ? 1 + 2 * nj : 1;
  const double dt = tab->dt;
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= (long long)m * n) return;
  const int row = (int)(e % m), col = (int)(e / m);
  const int blk = row / per, sub = row % per;
  const int j = blk / H, i = blk % H;
  const int jj = col / nj, k = col % nj;
  double val = 0.0;
  if (sub == 0) {
    const double g = grad[((size_t)j * H + i) * nj + k];
    if (jj <= i) val = -(g * (0.5 * dt * dt + ((i - jj) * dt) * dt));
    if (col == 0) {
      double gu = 0.0;
      for (int c = 0; c < n; ++c) {
        const int j2 = c / nj, k2 = c % nj;
        if (j2 <= i) gu += (grad[((size_t)j * H + i) * nj + k2] * (0.5 * dt * dt + ((i - j2) * dt) * dt)) * u[c];
      }
      const double margin = margin_is_D ? tab->obs[j].D : tab->obs[j].eps;
      binq[row] = (dist[(size_t)j * H + i] - margin) - gu;
    }
  } else {
    const int kk = (sub - 1) % nj, neg = (sub - 1) / nj;
    if (kk == k && jj <= i) val = neg ? -dt : dt;
    if (col == 0) binq[row] = neg ? lim[kk] + x0[nj + kk] : lim[kk] - x0[nj + kk];
  }
  Ainq[row + (size_t)m * col] = val;
}

cudaError_t launch_get_con_rows(const DevTables *tab, int H, int nj, int nobs, int has_lim, int margin_is_D,
                                const double *x0, const double *u, const double *lim, const double *dist,
                                const double *grad, double *Ainq, double *binq, int m, cudaStream_t s) {
  const long long total = (long long)m * H * nj;
  if (total <= 0) return cudaSuccess;
  k_get_con_rows<<<(int)((total + 255) / 256), 256, 0, s>>>(tab, H, nj, nobs, has_lim, margin_is_D, x0, u, lim, dist,
                                                              grad, Ainq, binq, m);
  return cudaGetLastError();
}

}  // namespace cfs
