// qp_warp.cuh -- the dual active-set QP of qp_core.cuh restated for ONE WARP per problem (k_warp.cu).
//
// Same method, same candidate rule, same tolerances and the same status codes as qp_solve<> in its cached-direction mode
// (every working-set member keeps z_w = QQ^-1 c_w'), but
//   * no CTA barrier anywhere: every phase change is a __syncwarp(), every reduction five shuffles;
//   * the primitives B_theta u / B_omega u are never stored: the violation scan computes them on the fly with warp prefix
//     sums (two consecutive waypoints per lane) and tests the velocity / control / obstacle rows straight from registers;
//   * sigma = c_p z_p and g_w = c_w z_p are dot products of a row (decoded on the fly, B_theta / B_omega in closed form)
//     with the candidate's direction -- no scratch for P z_p;
//   * the polish step is one line: the residual of S_W lambda = b is minus the slack of the active rows at u(lambda);
//   * the first WQ slots of the direction cache live in shared memory, the rest in a per-warp global slab (L2).
// Shared memory per problem: ~18-22 KB instead of 73.6 KB per CTA, so 9-12 problems are resident per SM, each on its own warp.
#pragma once
#include "cfs_kernels.cuh"

namespace cfs {

#define WQ_QS 16       // working sets of up to WQ_QS rows keep their inverse in shared memory (column-major, leading dimension WQ_QS)
#define WQ_QBIG 32     // ... beyond that, up to WQ_QBIG rows, in this warp's global slab (leading dimension WQ_QBIG, L2 resident)
#define WQ_QZ (WQ_QBIG + 1)  // direction slots (members + candidate): the first `zs` in shared memory, the rest in the slab
#define WQ_DEP_TOL 1e-8
#define FULLMASK 0xffffffffu

struct WDims {
  int n, H, OH, O, m, np, has_vel, has_bnd;
  double dt;
  const double *G;      // Gram operator (L2)
  const double *gdiag;  // sqrt(G_ii)
  const double *umax;   // MAX_input (global)
  const double *lim;    // velocity limits (global, CFS_MAXL)
  const double *qlim;   // LIM: joint position limits [qmax (NJ) | qmin (NJ)] (global), +-inf for a side without a limit
};

struct WView {  // this warp's shared-memory region
  double *th;     // n       theta part of x_
  double *uq;     // n       QP iterate u
  double *u0s;    // n       unconstrained minimiser
  double *ocoef;  // OH*NJ   -grad
  double *orhs;   // OH
  double *onrm;   // OH
  double *zc;     // zs*n    directions (also the gradient phase's scratch)
  double *M;      // WQ_QS*WQ_QS
  double *lam, *r, *g;  // WQ_QBIG+2
  double *x0s;    // 2*NJ (padded to 16)
  int *act;       // WQ_QBIG+2
  int *zslot;     // WQ_QZ+2
  unsigned char *inact;  // m
  double *zgl;    // global slab of this warp: (WQ_QZ - zs) * n directions, then WQ_QBIG*WQ_QBIG for the spilled inverse
  double *Mgl;
  int zs;         // direction slots in shared memory
  int qcap;       // working-set capacity in use (<= WQ_QBIG): beyond it the problem is handed to the heavy tier
};

__host__ __device__ inline size_t warp_scratch_doubles(int n, int nj, int zs) {
  const size_t a = (size_t)zs * n, b = (size_t)(2 * nj + 12) * 32;  // directions | sin/cos cache + kinematic prefix per lane
  return a > b ? a : b;
}

// lim: the 2n joint position rows' flags follow the inact byte map as bits (w_set_inact), so that the region grows by 2n / 8
// bytes only and the 12-warp CTA shape keeps fitting one SM
__host__ __device__ inline size_t warp_region_bytes(int n, int nj, int OH, int zs, bool lim = false) {
  size_t d = 3 * (size_t)n + (size_t)OH * (nj + 2) + warp_scratch_doubles(n, nj, zs) + WQ_QS * WQ_QS + 3 * (WQ_QBIG + 2) + 16;
  size_t b = d * sizeof(double) + sizeof(int) * (2 * WQ_QZ + 8) + (size_t)(OH + 4 * n) + (lim ? (size_t)(2 * n + 7) / 8 : 0);
  return (b + 15) / 16 * 16;
}

__device__ __forceinline__ WView warp_view(unsigned char *base, int n, int nj, int OH, int zs) {
  WView s;
  double *d = reinterpret_cast<double *>(base);
  s.th = d; d += n;
  s.uq = d; d += n;
  s.u0s = d; d += n;
  s.ocoef = d; d += (size_t)OH * nj;
  s.orhs = d; d += OH;
  s.onrm = d; d += OH;
  s.zc = d; d += warp_scratch_doubles(n, nj, zs);
  s.M = d; d += WQ_QS * WQ_QS;
  s.lam = d; d += WQ_QBIG + 2;
  s.r = d; d += WQ_QBIG + 2;
  s.g = d; d += WQ_QBIG + 2;
  s.x0s = d; d += 16;
  int *ip = reinterpret_cast<int *>(d);
  s.act = ip; ip += WQ_QZ + 2;
  s.zslot = ip; ip += WQ_QZ + 6;
  s.inact = reinterpret_cast<unsigned char *>(ip);
  s.zgl = nullptr;
  s.Mgl = nullptr;
  s.zs = zs;
  s.qcap = WQ_QS - 1;
  return s;
}

__host__ __device__ inline size_t warp_slab_doubles(int n, int zs) { return (size_t)(WQ_QZ - zs) * n + (size_t)WQ_QBIG * WQ_QBIG; }

__device__ __forceinline__ double *wz(const WView &s, int slot, int n) {
  return slot < s.zs ? s.zc + (size_t)slot * n : s.zgl + (size_t)(slot - s.zs) * n;
}

// inact flag of row cid: a byte per row, the LIM position rows (ids from OH + 4n) a bit each after the bytes.  Written by one
// lane between two __syncwarp()s.
template <bool LIM>
__device__ __forceinline__ bool w_inact(const WView &s, int m0, int cid) {
  if (LIM && cid >= m0) return (s.inact[m0 + ((cid - m0) >> 3)] >> ((cid - m0) & 7)) & 1;
  return s.inact[cid];
}
template <bool LIM>
__device__ __forceinline__ void w_set_inact(const WView &s, int m0, int cid, unsigned char v) {
  if (LIM && cid >= m0) {
    unsigned char *w = s.inact + m0 + ((cid - m0) >> 3);
    const unsigned char bit = (unsigned char)(1u << ((cid - m0) & 7));
    *w = v ? (unsigned char)(*w | bit) : (unsigned char)(*w & ~bit);
  } else {
    s.inact[cid] = v;
  }
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULLMASK, v, o);
  return v;
}

// minimum of (val, idx) over the lanes with idx >= 0; ties go to the lowest idx; every lane returns the same pair (and aux)
__device__ __forceinline__ void warp_argmin(double &val, int &idx, double &aux) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double ov = __shfl_xor_sync(FULLMASK, val, o);
    const int oi = __shfl_xor_sync(FULLMASK, idx, o);
    const double oa = __shfl_xor_sync(FULLMASK, aux, o);
    if (oi >= 0 && (idx < 0 || ov < val || (ov == val && oi < idx))) {
      val = ov;
      idx = oi;
      aux = oa;
    }
  }
}

__device__ __forceinline__ int w_wp_of(int cid, int H) {
  int i = cid;
  while (i >= H) i -= H;
  return i;
}

// joint position row (waypoint i + 1, joint k): +-theta <= qmax / -qmin, i.e. +-(B_theta u)(i,k) <= qmax - fm / fm - qmin with the
// free motion fm = theta0 + (i+1) dt omega0
__device__ __forceinline__ double w_pos_rhs(int e, int neg, int nj, const double *x0s, const double *qlim, double dt) {
  const int i = e / nj, k = e - i * nj;
  const double fm = x0s[k] + ((i + 1) * dt) * x0s[nj + k];
  return neg ? fm - __ldg(qlim + nj + k) : __ldg(qlim + k) - fm;
}

// LIM: ids OH + 4n + 2e + neg are the joint position rows of the theta primitive e = i NJ + k (DESIGN.md section 3d)
template <int NJ, bool LIM = false>
__device__ __forceinline__ double w_row_rhs(int cid, const WView &s, const WDims &P) {
  if (cid < P.OH) return s.orhs[cid];
  const int e = cid - P.OH, pr = e >> 1, neg = e & 1;
  if (pr < P.n) {
    const int k = pr % NJ;
    const double lim = __ldg(P.lim + k), w0 = s.x0s[NJ + k];
    return neg ? lim + w0 : lim - w0;
  }
  if (LIM && pr >= 2 * P.n) return w_pos_rhs(pr - 2 * P.n, neg, NJ, s.x0s, P.qlim, P.dt);
  return __ldg(P.umax + (pr - P.n));
}

// c_cid . vec for an n-vector in control space ([waypoint][joint]); the row is decoded on the fly:
//   obstacle row (j,i):        sum_{jj<=i} sum_k cv[k] (0.5+(i-jj)) dt^2 vec[jj,k]      (CFS_FANUC.m:121, B_theta blocks)
//   velocity row (i,k), +-:    +- dt sum_{jj<=i} vec[jj,k]                               (CFS_FANUC.m:126-129)
//   control row c, +-:         +- vec[c]                                                  (lb/ub of CFS_FANUC.m:85)
//   LIM, position row (i,k), +-: +- sum_{jj<=i} (0.5+(i-jj)) dt^2 vec[jj,k]
// Every lane returns the same value.  Not inlined (four call sites); every argument is a scalar, so nothing goes through
// local memory.
template <int NJ, bool LIM = false>
static __device__ __noinline__ double w_row_dot(int cid, const double *vec, const double *ocoef, int OH, int H, int n, double dt) {
  const int lane = threadIdx.x & 31;
  if (cid < OH) {
    const int i = w_wp_of(cid, H);
    const double *cv = ocoef + (size_t)cid * NJ;
    const int lim = (i + 1) * NJ;
    double acc = 0.0;
#pragma unroll 2
    for (int c = lane; c < lim; c += 32) {
      const int jj = c / NJ, k = c - jj * NJ;
      acc += (cv[k] * (0.5 * dt * dt + ((i - jj) * dt) * dt)) * vec[c];
    }
    return warp_sum(acc);
  }
  const int e = cid - OH, pr = e >> 1;
  const double sgn = (e & 1) ? -1.0 : 1.0;
  if (pr < n) {
    const int i = pr / NJ, k = pr - i * NJ;
    double acc = 0.0;
    for (int jj = lane; jj <= i; jj += 32) acc += vec[jj * NJ + k];
    return sgn * dt * warp_sum(acc);
  }
  if (LIM && pr >= 2 * n) {
    const int i = (pr - 2 * n) / NJ, k = (pr - 2 * n) - i * NJ;
    double acc = 0.0;
    for (int jj = lane; jj <= i; jj += 32) acc += (0.5 * dt * dt + ((i - jj) * dt) * dt) * vec[jj * NJ + k];
    return sgn * warp_sum(acc);
  }
  return sgn * vec[pr - n];
}
#define W_ROW_DOT(cid, vec) w_row_dot<NJ, LIM>(cid, vec, s.ocoef, P.OH, P.H, P.n, P.dt)

// primal recovery u = u0 - sum_w lambda_w z_w (n <= 32 * W_NC)
#define W_NC 10
__device__ __forceinline__ void w_refresh(const WView &s, const WDims &P, int q) {
  const int lane = threadIdx.x & 31, n = P.n;
  double acc[W_NC];
#pragma unroll
  for (int j = 0; j < W_NC; ++j) acc[j] = 0.0;
#pragma unroll 1
  for (int w = 0; w < q; ++w) {
    const double lw = s.lam[w];
    const double *z = wz(s, s.zslot[w], n) + lane;
#pragma unroll
    for (int j = 0; j < W_NC; ++j)
      if (lane + 32 * j < n) acc[j] += lw * z[32 * j];
  }
#pragma unroll
  for (int j = 0; j < W_NC; ++j)
    if (lane + 32 * j < n) s.uq[lane + 32 * j] = s.u0s[lane + 32 * j] - acc[j];
  __syncwarp();
}

// Inclusive warp prefix sums over the waypoints (two consecutive ones per lane, H <= 64): S1_i = sum_{j<=i} a_j at both
// waypoints of the lane, and T_i = sum_{j<i} S1_j at both.  Then (B_omega u)_i = dt S1_i and
// (B_theta u)_i = sum_{j<=i} (0.5 + (i-j)) dt^2 u_j = dt^2 (0.5 S1_i + T_i).
__device__ __forceinline__ void w_prefix2(double a0, double a1, double &s0, double &s1, double &t0, double &t1) {
  const int lane = threadIdx.x & 31;
  const double pr = a0 + a1;
  double inc = pr;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const double t = __shfl_up_sync(FULLMASK, inc, o);
    if (lane >= o) inc += t;
  }
  s0 = (inc - pr) + a0;
  s1 = inc;
  const double rr = s0 + s1;
  double inc2 = rr;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const double t = __shfl_up_sync(FULLMASK, inc2, o);
    if (lane >= o) inc2 += t;
  }
  t0 = inc2 - rr;
  t1 = t0 + s0;
}

// (1) most violated inactive row at the current uq, normalised by its QQ^-1 norm (same rule as qp_solve): returns its id
// (-1: none) and its slack.  B_theta u / B_omega u come from prefix sums held in registers (H <= 64: one pair of waypoints
// per lane, the NJ joints' scans interleaved); obstacles are taken two at a time.  While phase-A masking is on, the
// candidates of the masked levels are tracked in the same pass: when no unmasked row is violated, the next level is
// unmasked and its most violated row taken, exactly as a rescan with the same u would do.  LIM: the joint position rows
// are tested from the same registers (never masked).
template <int NJ, bool LIM = false>
__device__ __forceinline__ int w_scan(const WView &s, const WDims &P, int &masked, double &slack_out) {
  const int lane = threadIdx.x & 31, n = P.n, H = P.H, OH = P.OH, O = P.O;
  const double dt = P.dt, dt2 = dt * dt;
  double best = 0.0, bsl = 0.0, best2 = 0.0, bsl2 = 0.0, best3 = 0.0, bsl3 = 0.0;
  int bidx = -1, bidx2 = -1, bidx3 = -1;
  const int i0 = 2 * lane, i1 = i0 + 1;
  const bool v0 = i0 < H, v1 = i1 < H;
#pragma unroll 1
  for (int j0 = 0; j0 < (O > 0 ? O : 1); j0 += 2) {
    double accA0 = 0.0, accA1 = 0.0, accB0 = 0.0, accB1 = 0.0;
    const bool hasA = j0 < O, hasB = j0 + 1 < O;
    const double *cA = s.ocoef + ((size_t)j0 * H + i0) * NJ, *cB = cA + (size_t)H * NJ;
    // one joint's scans per trip: the unrolled form (the NJ independent scans interleaved) is ~1 000 instructions more
    // of the QP's hot loop and measured slower (DESIGN.md section 4b)
#pragma unroll 1
    for (int k = 0; k < NJ; ++k) {
      const double a0 = v0 ? s.uq[i0 * NJ + k] : 0.0, a1 = v1 ? s.uq[i1 * NJ + k] : 0.0;
      double s0, s1, t0, t1;
      w_prefix2(a0, a1, s0, s1, t0, t1);
      const double th0 = dt2 * (0.5 * s0 + t0), th1 = dt2 * (0.5 * s1 + t1);
      if (hasA) {
        if (v0) accA0 += cA[k] * th0;
        if (v1) accA1 += cA[NJ + k] * th1;
      }
      if (hasB) {
        if (v0) accB0 += cB[k] * th0;
        if (v1) accB1 += cB[NJ + k] * th1;
      }
      if (j0 == 0 && P.has_vel) {  // velocity rows +-(w0 + (B_omega u)(i,k)) <= lim   (CFS_FANUC.m:126-129)
        const double lim = __ldg(P.lim + k), w0 = s.x0s[NJ + k];
        const double tol = 1e-11 * (1.0 + lim);
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const double vw = w0 + dt * (h ? s1 : s0);
          const double sl = lim - fabs(vw);  // slack of the side that can be violated
          if ((h ? v1 : v0) && sl < -tol) {
            const int e = (h ? i1 : i0) * NJ + k, cu = OH + 2 * e + (vw < 0.0 ? 1 : 0);
            const double gd = __ldg(P.gdiag + n + e), sg = gd * gd;
            if (sg > 0.0 && !s.inact[cu]) {
              const double key = -(sl * sl) / sg;
              if (key < best || bidx < 0) { best = key; bidx = cu; bsl = sl; }
            }
          }
        }
      }
      if (LIM && j0 == 0) {  // position rows theta <= qmax, -theta <= -qmin: at most one side violated (qmin <= qmax)
        const double qhi = __ldg(P.qlim + k), qlo = __ldg(P.qlim + NJ + k), th00 = s.x0s[k], w0 = s.x0s[NJ + k];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int i = h ? i1 : i0;
          const double fm = th00 + ((i + 1) * dt) * w0, th = h ? th1 : th0;
          const double hi = qhi - fm, lo = fm - qlo, up = hi - th, dn = lo + th;
          const bool neg = dn < up;
          const double sl = neg ? dn : up;
          if ((h ? v1 : v0) && sl < -1e-11 * (1.0 + fabs(neg ? lo : hi))) {
            const int e = i * NJ + k, cu = OH + 4 * n + 2 * e + (neg ? 1 : 0);
            const double gd = __ldg(P.gdiag + e), sg = gd * gd;
            if (sg > 0.0 && !w_inact<LIM>(s, OH + 4 * n, cu)) {
              const double key = -(sl * sl) / sg;
              if (key < best || bidx < 0) { best = key; bidx = cu; bsl = sl; }
            }
          }
        }
      }
    }
    // obstacle rows of this pair of obstacles at the lane's two waypoints
#pragma unroll
    for (int r4 = 0; r4 < 4; ++r4) {
      const bool second = r4 & 1, obsB = r4 >> 1;
      if (obsB ? !hasB : !hasA) continue;
      if (!(second ? v1 : v0)) continue;
      const int cid = (j0 + (obsB ? 1 : 0)) * H + (second ? i1 : i0);
      const double sg = s.onrm[cid];
      const int lvl = s.inact[cid];
      if (lvl == 1 || !(sg > 0.0)) continue;
      const double val = obsB ? (second ? accB1 : accB0) : (second ? accA1 : accA0);
      const double rhs = s.orhs[cid];
      const double sl = rhs - val;
      if (sl < -1e-11 * (1.0 + fabs(rhs))) {
        const double key = -(sl * sl) / sg;
        if (lvl == 0) {
          if (key < best || bidx < 0) { best = key; bidx = cid; bsl = sl; }
        } else if (lvl == 2) {
          if (key < best2 || bidx2 < 0) { best2 = key; bidx2 = cid; bsl2 = sl; }
        } else {
          if (key < best3 || bidx3 < 0) { best3 = key; bidx3 = cid; bsl3 = sl; }
        }
      }
    }
  }
  if (P.has_bnd) {  // control rows +-u <= MAX_input
#pragma unroll 1
    for (int c = lane; c < n; c += 32) {
      const double uv = s.uq[c], um = __ldg(P.umax + c);
      const double sl = um - fabs(uv);
      if (sl < -1e-11 * (1.0 + um)) {
        const int cu = OH + 2 * (n + c) + (uv < 0.0 ? 1 : 0);
        const double gd = __ldg(P.gdiag + 2 * n + c), sg = gd * gd;
        if (sg > 0.0 && !s.inact[cu]) {
          const double key = -(sl * sl) / sg;
          if (key < best || bidx < 0) { best = key; bidx = cu; bsl = sl; }
        }
      }
    }
  }
  warp_argmin(best, bidx, bsl);
  while (bidx < 0 && masked) {  // this phase is feasible: unmask the next level, same working set
    const int lvl = masked == 2 ? 2 : 3;
#pragma unroll 1
    for (int cid = lane; cid < OH; cid += 32)
      if (s.inact[cid] == lvl) s.inact[cid] = 0;
    if (lvl == 2) {
      warp_argmin(best2, bidx2, bsl2);
      bidx = bidx2;
      bsl = bsl2;
    } else {
      warp_argmin(best3, bidx3, bsl3);
      bidx = bidx3;
      bsl = bsl3;
    }
    --masked;
    __syncwarp();
  }
  slack_out = bsl;
  return bidx;
}

// Phase A of every QP (see qp_mask_antiparallel in qp_core.cuh): mask all obstacle rows except the most anti-parallel
// consecutive pair (level 2: every pair with cos < -0.9, level 3: the rest).  Returns the number of masking levels set.
template <int NJ>
__device__ __forceinline__ int w_mask_antiparallel(const WView &s, const WDims &P) {
  const int lane = threadIdx.x & 31, OH = P.OH, H = P.H;
  double best = 0.0, aux = 0.0;
  int bidx = -1;
  unsigned apbits = 0;  // bit j: rows (cid, cid+1), cid = lane + 32 j, are anti-parallel
#pragma unroll 1
  for (int cid = lane, j = 0; cid < OH; cid += 32, ++j) {
    if (w_wp_of(cid, H) == H - 1) continue;  // the pair must belong to the same obstacle
    const double *a = s.ocoef + (size_t)cid * NJ, *b = a + NJ;
    double ab = 0.0, aa = 0.0, bb = 0.0;
#pragma unroll
    for (int k = 0; k < NJ; ++k) {
      ab += a[k] * b[k];
      aa += a[k] * a[k];
      bb += b[k] * b[k];
    }
    if (ab < 0.0 && ab * ab > 0.81 * aa * bb) {  // cos < -0.9
      apbits |= 1u << (j & 31);
      const double cs = ab / sqrt(aa * bb);
      if (bidx < 0 || cs < best) {
        best = cs;
        bidx = cid;
      }
    }
  }
  warp_argmin(best, bidx, aux);
  if (bidx < 0) return 0;
#pragma unroll 1
  for (int cid = lane; cid < OH; cid += 32) s.inact[cid] = 3;
  __syncwarp();
#pragma unroll 1
  for (int cid = lane, j = 0; cid < OH; cid += 32, ++j)
    if ((apbits >> (j & 31)) & 1u) {
      s.inact[cid] = 2;
      s.inact[cid + 1] = 2;
    }
  __syncwarp();
  if (lane == 0) {
    s.inact[bidx] = 0;
    s.inact[bidx + 1] = 0;
  }
  __syncwarp();
  return 2;
}

// Solves  min 1/2 u'QQ u + ff'u  s.t. the rows in (s.ocoef, s.orhs, lim, umax), starting from u0s.  On return (status 0)
// s.uq holds the optimum, s.lam / s.act / q the multipliers and the working set.
// status: 0 optimal, 2 infeasible, 3 numerical, 4 escalate (step_cap exceeded / working set outgrew the direction slots).
template <int NJ, bool LIM = false>
__device__ __forceinline__ int wqp_solve(const WView &s, const WDims &P, double cost0, double fupper, int step_cap, int masked,
                                         int &q_out, int &steps_out, int &qmax_seen) {
  const int lane = threadIdx.x & 31, n = P.n, OH = P.OH;
  int q = 0, status = -1, steps = 0;
  bool polished = false;
#pragma unroll 1
  for (int e = lane; e <= WQ_QZ; e += 32) s.zslot[e] = e;
  __syncwarp();
  double fval = cost0;
  const int max_steps = 20 * (P.m + n) + 100;
  double *Mp = s.M;  // working-set inverse: shared memory up to WQ_QS rows, then this warp's global slab
  int ldm = WQ_QS;
  while (status < 0) {
    w_refresh(s, P, q);
    double sp;
    const int p = w_scan<NJ, LIM>(s, P, masked, sp);
    if (p < 0) {
      if (q == 0 || polished || (steps <= 6 && q <= 6)) {
        status = 0;
        break;
      }
      // polish: one step of iterative refinement on S_W lambda = b; its residual is minus the slack of the active rows
#pragma unroll 1
      for (int w = 0; w < q; ++w) {
        const int cw = s.act[w];
        const double val = W_ROW_DOT(cw, s.uq) - w_row_rhs<NJ, LIM>(cw, s, P);
        if (lane == 0) s.g[w] = val;
      }
      __syncwarp();
#pragma unroll 1
      for (int w = lane; w < q; w += 32) {
        double acc = 0.0;
#pragma unroll 4
        for (int c = 0; c < q; ++c) acc += Mp[w + (size_t)ldm * c] * s.g[c];
        s.lam[w] += acc;
      }
      __syncwarp();
      polished = true;
      continue;
    }
    polished = false;
    if (q > s.qcap) {  // no slot left for the candidate's direction: the heavy tier redoes this iteration
      status = 4;
      break;
    }
    // candidate direction z_p = QQ^-1 c_p': one pass over <= NJ rows of the control block of G
    double *zp = wz(s, s.zslot[q], n);
    {
      const double *__restrict__ Gu = P.G + 2 * n;
      if (p < OH) {
        const double *cv = s.ocoef + (size_t)p * NJ;
        const double *__restrict__ G0 = Gu + (size_t)(w_wp_of(p, P.H) * NJ) * P.np;
        double cvr[NJ];
#pragma unroll
        for (int k = 0; k < NJ; ++k) cvr[k] = cv[k];
#pragma unroll 2
        for (int c = lane; c < n; c += 32) {
          double acc = 0.0;
#pragma unroll
          for (int k = 0; k < NJ; ++k) acc += cvr[k] * G0[(size_t)k * P.np + c];
          zp[c] = acc;
        }
      } else {
        const int e = p - OH;
        const double coef = (e & 1) ? -1.0 : 1.0;
        // primitive row of G: omega / control rows n + pr, LIM position rows pr - 2n (the theta block)
        const double *__restrict__ G0 = Gu + (size_t)((LIM && (e >> 1) >= 2 * n) ? (e >> 1) - 2 * n : n + (e >> 1)) * P.np;
#pragma unroll 4
        for (int c = lane; c < n; c += 32) zp[c] = coef * G0[c];
      }
    }
    __syncwarp();
    // sigma = c_p z_p and g_w = c_w z_p: one call site, the candidate rides along as "member q"
    double sigma = 0.0;
#pragma unroll 1
    for (int w = 0; w <= q; ++w) {
      const double val = W_ROW_DOT(w < q ? s.act[w] : p, zp);
      if (w < q) {
        if (lane == 0) s.g[w] = val;
      } else {
        sigma = val;
      }
    }
    __syncwarp();
    double lam_p = 0.0;
    // (2) bring row p into the working set (rows of the inverse are strided over the lanes)
    for (;;) {
      if (++steps > max_steps) {
        status = 3;
        break;
      }
      if (steps > step_cap) {
        status = 4;
        break;
      }
      double part = 0.0, t1 = INFINITY, aux = 0.0;
      int l = -1;
#pragma unroll 1
      for (int w = lane; w < q; w += 32) {
        double rw = 0.0;
#pragma unroll 4
        for (int c = 0; c < q; ++c) rw += Mp[w + (size_t)ldm * c] * s.g[c];
        s.r[w] = rw;
        part += s.g[w] * rw;
        if (rw > 0.0) {
          const double tt = s.lam[w] / rw;
          if (l < 0 || tt < t1) {
            t1 = tt;
            l = w;
          }
        }
      }
      const double delta = sigma - warp_sum(part);
      warp_argmin(t1, l, aux);
      if (l < 0) t1 = INFINITY;
      if (!(delta == delta) || !(sigma == sigma)) {
        status = 3;
        break;
      }
      const bool dependent = !(delta > WQ_DEP_TOL * sigma) || q >= n;
      double t2 = INFINITY;
      if (!dependent) {
        t2 = -sp / delta;
        if (t2 < 0.0) t2 = 0.0;
      }
      if (l < 0 && dependent) {
        status = 2;
        break;
      }
      const bool full = (t2 <= t1);
      const double t = full ? t2 : t1;
      if (!dependent) {
        fval += t * delta * (0.5 * t + lam_p);
        sp += t * delta;
      }
      if (fval > fupper) {
        status = 2;
        break;
      }
#pragma unroll 1
      for (int w = lane; w < q; w += 32) s.lam[w] -= t * s.r[w];
      lam_p += t;
      __syncwarp();
      if (full) {
        if (q + 1 > WQ_QBIG) {
          status = 4;
          break;
        }
        if (q + 1 > WQ_QS && Mp == s.M) {  // the inverse outgrows shared memory: move it to the slab
#pragma unroll 1
          for (int e = lane; e < q * q; e += 32) {
            const int c = e / q, rr = e - c * q;
            s.Mgl[rr + (size_t)WQ_QBIG * c] = s.M[rr + WQ_QS * c];
          }
          Mp = s.Mgl;
          ldm = WQ_QBIG;
          __syncwarp();
        }
        // bordered inverse [[M + r r'/d, -r/d], [-r'/d, 1/d]]
        const double id = 1.0 / delta;
#pragma unroll 1
        for (int c = 0; c <= q; ++c) {
          const double rc = c < q ? s.r[c] : 0.0;
#pragma unroll 1
          for (int rr = lane; rr <= q; rr += 32) {
            double val;
            if (rr < q && c < q)
              val = Mp[rr + (size_t)ldm * c] + s.r[rr] * (rc * id);
            else if (rr == q && c == q)
              val = id;
            else
              val = -(rr < q ? s.r[rr] : rc) * id;
            Mp[rr + (size_t)ldm * c] = val;
          }
        }
        if (lane == 0) {
          s.act[q] = p;
          s.lam[q] = lam_p;
          w_set_inact<LIM>(s, OH + 4 * n, p, 1);
        }
        ++q;
        if (q > qmax_seen) qmax_seen = q;
        __syncwarp();
        break;
      }
      // drop member l: M <- M - M(:,l) M(l,:)/M(l,l), then move the last member into slot l (s.r holds column l meanwhile)
      {
        const int last = q - 1;
#pragma unroll 1
        for (int w = lane; w < q; w += 32) s.r[w] = Mp[w + (size_t)ldm * l];
        __syncwarp();
        const double ip = 1.0 / s.r[l];
#pragma unroll 1
        for (int c = 0; c < q; ++c) {
          const double gc = s.r[c] * ip;
#pragma unroll 1
          for (int w = lane; w < q; w += 32) Mp[w + (size_t)ldm * c] -= s.r[w] * gc;
        }
        __syncwarp();
        if (l != last) {
#pragma unroll 1
          for (int w = lane; w < q; w += 32) Mp[w + (size_t)ldm * l] = Mp[w + (size_t)ldm * last];
          __syncwarp();
#pragma unroll 1
          for (int w = lane; w < q; w += 32) Mp[l + (size_t)ldm * w] = Mp[last + (size_t)ldm * w];
        }
        if (lane == 0) {
          w_set_inact<LIM>(s, OH + 4 * n, s.act[l], 0);
          s.act[l] = s.act[last];
          s.lam[l] = s.lam[last];
          s.g[l] = s.g[last];
          const int freed = s.zslot[l];
          s.zslot[l] = s.zslot[last];
          s.zslot[last] = s.zslot[q];
          s.zslot[q] = freed;
        }
        --q;
        __syncwarp();
      }
    }
  }
  q_out = q;
  steps_out = steps;
  return status;
}

}  // namespace cfs
