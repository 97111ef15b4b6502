// qp_core.cuh -- the batched dual active-set QP core shared by the lock-step kernel (k_qp.cu) and the fused persistent
// kernel (k_fused.cu).  See k_qp.cu for the design notes.
#pragma once
#include "cfs_kernels.cuh"

namespace cfs {

#define QP_THREADS 128   // lock-step kernel / bulk tier of the fused kernel
#define QP_DEP_TOL 1e-8
#define QP_QS 48          // working sets up to QP_QS keep their inverse in shared memory
#define QP_SMALL_T 20     // term lists up to this length refresh all 3n primitives directly from G

struct QpView {  // decoded shared-memory layout
  double *v;       // np
  double *ocoef;   // OH*nj   (-g)
  double *orhs;    // OH
  double *onrm;    // OH      scan normalisation of every obstacle row: sum_k c_k^2 G_ii (diagonal proxy of c QQ^-1 c')
  double *lam;     // n+2
  double *r;       // n+2
  double *g;       // n+2
  double *red;     // 16
  double *tcoef;   // TMAX    coefficient of each active term
  double *twgt;    // TMAX    lambda_owner * coefficient
  double *Msm;     // QP_QS*QP_QS
  double *lim;     // 8: velocity limits; lim layouts: then qmax | qmin | theta0 (8 each) of the joint position rows
  double *w0;      // 8: initial joint velocities
  int *act;        // n+2
  int *toff;       // n+3     first term of each working-set member
  int *trow;       // TMAX    primitive row of each active term
  int *towner;     // TMAX
  int *ctl;        // 8
  unsigned char *inact;  // m
  double *v0s;     // np      v at the unconstrained minimiser (per problem)
  double *gns;     // 3n      G_ii of every primitive row (per kernel)
  double *ums;     // n       MAX_input (per kernel)
  double *pscr;    // QP_THREADS  partial sums of the polish residual
  double *zc;      // QZ*n   cached directions z_w = QQ^-1 c_w' of the working-set members + the candidate (bulk tier)
  int *zslot;      // QZ+1   physical slot of member w; zslot[q] is the candidate's slot
  double *yp;      // 2n     B_theta z_p | B_omega z_p of the candidate (cached mode)
};

#define QP_NOFF 26
// qz > 0: "cached" layout of the fused bulk tier -- the working set holds at most qz-1 rows, every member's direction
// z_w (n doubles) stays in shared memory, and the flat term lists of the G-based refresh are not needed.
// lim: layout of the joint-limit instantiations (m then counts the 2n position rows too)
__host__ __device__ inline size_t qp_smem_layout(int n, int nj, int OH, int m, size_t *off /*[QP_NOFF]*/, int qs = QP_QS,
                                                  int nt = QP_THREADS, int qz = 0, bool lim = false) {
  size_t o = 0;
  const int np = 3 * n;
  const int tmax = qz ? 0 : nj * OH + n + 2;
  const int nw = qz ? qz + 2 : n + 2;  // capacity of the per-member arrays
  // [zc | Msm | v | tcoef | twgt | lam | r | g] first and contiguous: all of it is dead while the fused kernel runs its
  // gradient phase, which aliases its scratch onto this span (qp_scratch_span()).
  off[23] = o; o += sizeof(double) * (size_t)qz * n;
  off[25] = o; o += sizeof(double) * (size_t)(qz ? 2 * n : 0);
  off[10] = o; o += sizeof(double) * qs * qs;
  off[0] = o; o += sizeof(double) * np;
  off[8] = o; o += sizeof(double) * tmax;
  off[9] = o; o += sizeof(double) * tmax;
  off[4] = o; o += sizeof(double) * nw;
  off[5] = o; o += sizeof(double) * nw;
  off[6] = o; o += sizeof(double) * nw;
  off[1] = o; o += sizeof(double) * (size_t)OH * nj;
  off[2] = o; o += sizeof(double) * OH;
  off[3] = o; o += sizeof(double) * OH;
  off[7] = o; o += sizeof(double) * 64;
  off[11] = o; o += sizeof(double) * (lim ? 32 : 8);
  off[12] = o; o += sizeof(double) * 8;
  off[13] = o; o += sizeof(int) * nw;
  off[14] = o; o += sizeof(int) * (nw + 2);
  off[15] = o; o += sizeof(int) * tmax;
  off[16] = o; o += sizeof(int) * tmax;
  off[17] = o; o += sizeof(int) * 8;
  off[24] = o; o += sizeof(int) * (size_t)(qz ? qz + 2 : 0);
  off[18] = o; o += (size_t)((m + 15) / 16) * 16;
  o = (o + 15) / 16 * 16;
  off[19] = o; o += sizeof(double) * np;
  off[20] = o; o += sizeof(double) * 3 * n;
  off[21] = o; o += sizeof(double) * n;
  off[22] = o; o += sizeof(double) * nt;
  return (o + 15) / 16 * 16;
}

__host__ __device__ inline size_t qp_scratch_span(int n, int nj, int OH, int qs = QP_QS, int qz = 0) {  // bytes of the leading dead-during-gradient span
  const int tmax = qz ? 0 : nj * OH + n + 2;
  const int nw = qz ? qz + 2 : n + 2;
  return sizeof(double) * ((size_t)qz * n + (size_t)(qz ? 2 * n : 0) + (size_t)qs * qs + 3 * n + 2 * (size_t)tmax + 3 * (size_t)nw);
}

__device__ __forceinline__ QpView qp_view(unsigned char *smem_raw, int n, int nj, int OH, int m, int qs = QP_QS,
                                          int nt = QP_THREADS, int qz = 0, bool lim = false) {
  QpView s;
  size_t off[QP_NOFF];
  qp_smem_layout(n, nj, OH, m, off, qs, nt, qz, lim);
  s.zc = reinterpret_cast<double *>(smem_raw + off[23]);
  s.zslot = reinterpret_cast<int *>(smem_raw + off[24]);
  s.yp = reinterpret_cast<double *>(smem_raw + off[25]);
  s.v = reinterpret_cast<double *>(smem_raw + off[0]);
  s.ocoef = reinterpret_cast<double *>(smem_raw + off[1]);
  s.orhs = reinterpret_cast<double *>(smem_raw + off[2]);
  s.onrm = reinterpret_cast<double *>(smem_raw + off[3]);
  s.lam = reinterpret_cast<double *>(smem_raw + off[4]);
  s.r = reinterpret_cast<double *>(smem_raw + off[5]);
  s.g = reinterpret_cast<double *>(smem_raw + off[6]);
  s.red = reinterpret_cast<double *>(smem_raw + off[7]);
  s.tcoef = reinterpret_cast<double *>(smem_raw + off[8]);
  s.twgt = reinterpret_cast<double *>(smem_raw + off[9]);
  s.Msm = reinterpret_cast<double *>(smem_raw + off[10]);
  s.lim = reinterpret_cast<double *>(smem_raw + off[11]);
  s.w0 = reinterpret_cast<double *>(smem_raw + off[12]);
  s.act = reinterpret_cast<int *>(smem_raw + off[13]);
  s.toff = reinterpret_cast<int *>(smem_raw + off[14]);
  s.trow = reinterpret_cast<int *>(smem_raw + off[15]);
  s.towner = reinterpret_cast<int *>(smem_raw + off[16]);
  s.ctl = reinterpret_cast<int *>(smem_raw + off[17]);
  s.inact = smem_raw + off[18];
  s.v0s = reinterpret_cast<double *>(smem_raw + off[19]);
  s.gns = reinterpret_cast<double *>(smem_raw + off[20]);
  s.ums = reinterpret_cast<double *>(smem_raw + off[21]);
  s.pscr = reinterpret_cast<double *>(smem_raw + off[22]);
  return s;
}

// ---- constraint rows ------------------------------------------------------------------------------------------
// cid in [0,OH): obstacle row (j,i), cid = j*H+i: nj terms on the theta primitives of waypoint i, coefficients ocoef[cid*nj+k]
// cid >= OH: e = cid-OH, primitive pr = e>>1 in [0,2n) (omega primitives 0..n-1, controls n..2n-1), sign bit e&1
//            (0: +row <= hi, 1: -row <= lo).  Velocity rows: CFS_FANUC.m:126-129; control rows: lb/ub of CFS_FANUC.m:85.
//            LIM (the joint-limit instantiations): pr in [2n,3n) is the theta primitive pr-2n, the joint position rows
//            theta <= qmax / -theta <= -qmin (DESIGN.md section 3d).
struct Desc {
  int nterm;
  int row0;          // first primitive row; terms are consecutive rows
  double coef;       // single-term coefficient (+-1) when nterm == 1
  const double *cv;  // coefficient vector when nterm > 1
};

struct QpDims {
  int n, nj, H, np, OH, m, has_vel, has_bnd;
  const double *G;     // Gram operator (L2 resident)
  const double *umax;  // MAX_input (shared memory copy)
  double *Mgl;         // this CTA's spill slab for the working-set inverse
  int ldg;
  double dt;
};

__device__ __forceinline__ int wp_of(int cid, int H) {  // waypoint of an obstacle row (few obstacles: no division)
  int i = cid;
  while (i >= H) i -= H;
  return i;
}

template <bool LIM = false>
__device__ __forceinline__ Desc decode(int cid, const QpDims &P, const double *ocoef) {
  Desc d;
  if (cid < P.OH) {
    d.nterm = P.nj;
    d.row0 = wp_of(cid, P.H) * P.nj;
    d.coef = 0.0;
    d.cv = ocoef + (size_t)cid * P.nj;
  } else {
    const int e = cid - P.OH;
    d.nterm = 1;
    d.row0 = (LIM && (e >> 1) >= 2 * P.n) ? (e >> 1) - 2 * P.n : P.n + (e >> 1);
    d.coef = (e & 1) ? -1.0 : 1.0;
    d.cv = nullptr;
  }
  return d;
}

// c_a QQ^-1 c_b' as a bilinear form over G
template <bool LIM = false>
static __device__ __noinline__ double gram(int ca, int cb, const QpDims &P, const double *ocoef) {
  const Desc a = decode<LIM>(ca, P, ocoef), b = decode<LIM>(cb, P, ocoef);
  const double *__restrict__ G = P.G;
  if (a.nterm == 1 && b.nterm == 1) return a.coef * b.coef * G[(size_t)a.row0 * P.np + b.row0];
  double s = 0.0;
#pragma unroll 1
  for (int k = 0; k < a.nterm; ++k) {
    const double ck = a.cv ? a.cv[k] : a.coef;
    const double *Gr = G + (size_t)(a.row0 + k) * P.np + b.row0;
    double t = 0.0;
#pragma unroll 6
    for (int l = 0; l < b.nterm; ++l) t += (b.cv ? b.cv[l] : b.coef) * Gr[l];  // independent L2 loads in flight
    s += ck * t;
  }
  return s;
}

template <int NJ, bool LIM = false>
__device__ __forceinline__ double prim_rhs(int pr, int neg, const QpDims &P, const QpView &s) {
  if (pr < P.n) {
    const int k = NJ ? pr % NJ : pr % P.nj;
    return neg ? s.lim[k] + s.w0[k] : s.lim[k] - s.w0[k];
  }
  if (LIM && pr >= 2 * P.n) {  // free motion fm = theta0 + (i+1) dt omega0: qmax - fm / fm - qmin
    const int nj = NJ ? NJ : P.nj, i = (pr - 2 * P.n) / nj, k = (pr - 2 * P.n) - i * nj;
    const double fm = s.lim[24 + k] + ((i + 1) * P.dt) * s.w0[k];
    return neg ? fm - s.lim[16 + k] : s.lim[8 + k] - fm;
  }
  return P.umax[pr - P.n];
}

// slack = rhs - c u from the primitive values in `v`; with v = v0s this is minus the violation at the unconstrained minimiser
template <int NJ, bool LIM = false>
static __device__ __noinline__ double slack_at(int cid, const QpDims &P, const QpView &s, const double *v) {
  if (cid < P.OH) {
    const double *c = s.ocoef + (size_t)cid * P.nj;
    const double *vv = v + wp_of(cid, P.H) * P.nj;
    double val = 0.0;
#pragma unroll 1
    for (int k = 0; k < P.nj; ++k) val += c[k] * vv[k];
    return s.orhs[cid] - val;
  }
  const int e = cid - P.OH, pr = e >> 1, neg = e & 1;
  const double vv = (LIM && pr >= 2 * P.n) ? v[pr - 2 * P.n] : v[P.n + pr];
  return prim_rhs<NJ, LIM>(pr, neg, P, s) - (neg ? -vv : vv);
}

// ---- block reductions (NT threads): warp shuffles, one shared-memory exchange, second stage again by shuffles -------
template <int NT>
static __device__ __noinline__ void block_argmin(double &val, int &idx, double *red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double ov = __shfl_xor_sync(0xffffffffu, val, o);
    const int oi = __shfl_xor_sync(0xffffffffu, idx, o);
    if (oi >= 0 && (idx < 0 || ov < val || (ov == val && oi < idx))) {
      val = ov;
      idx = oi;
    }
  }
  constexpr int NW = NT / 32;
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __syncthreads();  // protect red from the previous use
  if (lane == 0) {
    red[2 * w] = val;
    reinterpret_cast<int *>(red + 2 * w + 1)[0] = idx;
  }
  __syncthreads();
  val = lane < NW ? red[2 * lane] : 0.0;
  idx = lane < NW ? reinterpret_cast<int *>(red + 2 * lane + 1)[0] : -1;
#pragma unroll
  for (int o = NW / 2; o > 0; o >>= 1) {
    const double ov = __shfl_xor_sync(0xffffffffu, val, o);
    const int oi = __shfl_xor_sync(0xffffffffu, idx, o);
    if (oi >= 0 && (idx < 0 || ov < val || (ov == val && oi < idx))) {
      val = ov;
      idx = oi;
    }
  }
  val = __shfl_sync(0xffffffffu, val, 0);  // every thread of the CTA leaves with the same (val, idx), NaNs included
  idx = __shfl_sync(0xffffffffu, idx, 0);
}

template <int NT>
static __device__ __noinline__ double block_sum(double val, double *red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) val += __shfl_xor_sync(0xffffffffu, val, o);
  constexpr int NW = NT / 32;
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __syncthreads();
  if (lane == 0) red[w] = val;
  __syncthreads();
  double s = lane < NW ? red[lane] : 0.0;
#pragma unroll
  for (int o = NW / 2; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  return __shfl_sync(0xffffffffu, s, 0);
}

#ifdef PF_GRAD_DETAIL  // dev build: slots 0-4 = gradient sub-phases, every QP phase lands in slot 5
#define QPF(k) 5
#else
#define QPF(k) k
#endif
#define PF_START() do { if (prof && tid == 0) tck = clock64(); } while (0)
#define PF_ADD(k) do { if (prof && tid == 0) { const long long now_ = clock64(); pf[k] += now_ - tck; tck = now_; } } while (0)

// (0) primal recovery from the multipliers: v = v0 - G (C_W' lambda).  The n control entries come from G (one pass over
// the flat list of active (primitive row, weight) terms, or, once the list is longer than n, through the control-space
// vector y = P' z and QQ^-1 y); B_theta u and B_omega u follow in closed form.
template <int NT, int UNR>
static __device__ __noinline__ void qp_refresh(const QpView &s, const QpDims &P, int q) {
  const int tid = threadIdx.x, n = P.n, nj = P.nj, np = P.np;
  const double dt = P.dt;
  const int T = s.toff[q];
#pragma unroll 1
  for (int t = tid; t < T; t += NT) s.twgt[t] = s.lam[s.towner[t]] * s.tcoef[t];
  __syncthreads();
  if (T <= QP_SMALL_T) {  // short term list: all 3n primitives straight from G, three entries x T loads in flight
    const double *__restrict__ G = P.G;
#pragma unroll 1
    for (int pi = tid; pi < np; pi += 3 * NT) {
      double a0 = 0.0, a1 = 0.0, a2 = 0.0;
      const bool k1 = pi + NT < np, k2 = pi + 2 * NT < np;
#pragma unroll 4
      for (int t = 0; t < T; ++t) {
        const double *g = G + (size_t)s.trow[t] * np + pi;
        const double w = s.twgt[t];
        a0 += w * g[0];
        if (k1) a1 += w * g[NT];
        if (k2) a2 += w * g[2 * NT];
      }
      s.v[pi] = s.v0s[pi] - a0;
      if (k1) s.v[pi + NT] = s.v0s[pi + NT] - a1;
      if (k2) s.v[pi + 2 * NT] = s.v0s[pi + 2 * NT] - a2;
    }
    __syncthreads();
    return;
  }
  const double *__restrict__ Gu = P.G + 2 * n;  // control block of every primitive row
  if (T <= n && (n & 1) == 0 && n / 2 <= NT) {
    // column pairs (16-byte loads) x up to two term groups; partial sums per column combined through s.g / s.r
    const int npair = n / 2, ngrp = NT / npair >= 2 ? 2 : 1;
    const int grp = tid / npair, pair = tid - grp * npair;
    if (grp < ngrp) {
      double a0 = 0.0, a1 = 0.0;
#pragma unroll UNR
      for (int t = grp; t < T; t += ngrp) {
        const double2 gq = *reinterpret_cast<const double2 *>(Gu + (size_t)s.trow[t] * np + 2 * pair);
        const double w = s.twgt[t];
        a0 += w * gq.x;
        a1 += w * gq.y;
      }
      double *dst = grp ? s.r : s.g;
      dst[2 * pair] = a0;
      dst[2 * pair + 1] = a1;
    }
    __syncthreads();
#pragma unroll 1
    for (int c = tid; c < n; c += NT) s.v[2 * n + c] = s.v0s[2 * n + c] - (ngrp == 2 ? s.g[c] + s.r[c] : s.g[c]);
  } else if (T <= n) {
#pragma unroll 1
    for (int c = tid; c < n; c += NT) {
      double acc = 0.0;
#pragma unroll 8
      for (int t = 0; t < T; ++t) acc += s.twgt[t] * Gu[(size_t)s.trow[t] * np + c];
      s.v[2 * n + c] = s.v0s[2 * n + c] - acc;
    }
  } else {
    // z = C_W' lambda scattered on the primitive index space (into v), y = P' z (into g), u = u0 - QQ^-1 y
#pragma unroll 1
    for (int e = tid; e < np; e += NT) s.v[e] = 0.0;
    __syncthreads();
#pragma unroll 1
    for (int t = tid; t < T; t += NT) atomicAdd(&s.v[s.trow[t]], s.twgt[t]);
    __syncthreads();
#pragma unroll 1
    for (int e = tid; e < n; e += NT) {
      const int j = e / nj, k = e - j * nj;
      double acc = s.v[2 * n + e];
#pragma unroll 1
      for (int i = j; i * nj < n; ++i)
        acc += (0.5 * dt * dt + ((i - j) * dt) * dt) * s.v[i * nj + k] + dt * s.v[n + i * nj + k];
      s.g[e] = acc;
    }
    __syncthreads();
    const double *__restrict__ Hi = Gu + (size_t)2 * n * np;  // QQ^-1 = control rows x control columns of G
#pragma unroll 1
    for (int c = tid; c < n; c += NT) {
      double acc = 0.0;
#pragma unroll 8
      for (int r = 0; r < n; ++r) acc += s.g[r] * Hi[(size_t)r * np + c];
      s.v[2 * n + c] = s.v0s[2 * n + c] - acc;
    }
  }
  __syncthreads();
#pragma unroll 1
  for (int e = tid; e < n; e += NT) {  // B_theta u and B_omega u in closed form
    const int i = e / nj, k = e - i * nj;
    double at = 0.0, aw = 0.0;
#pragma unroll 4
    for (int j = 0; j <= i; ++j) {
      const double uj = s.v[2 * n + j * nj + k];
      at += (0.5 * dt * dt + ((i - j) * dt) * dt) * uj;
      aw += dt * uj;
    }
    s.v[e] = at;
    s.v[n + e] = aw;
  }
  __syncthreads();
}

// ---- cached-direction mode (fused bulk tier) ------------------------------------------------------------------------
// Every working-set member w keeps z_w = QQ^-1 c_w' (n doubles, one pass over <= nj rows of G when the row becomes the
// candidate) in shared memory.  Then nothing inside a dual step touches L2 any more:
//   primal recovery   u = u0 - sum_w lambda_w z_w,  B_theta u and B_omega u in closed form
//   sigma, g_w        e_p'(P z_p), e_w'(P z_p): closed-form partial sums over the candidate's direction

// B_theta u and B_omega u of the control vector u (n entries, [waypoint][joint]) by warp-level prefix sums: one warp per
// joint, two consecutive waypoints per lane.  With S1_i = sum_{j<=i} u_j:
//   (B_omega u)_i = dt S1_i,   (B_theta u)_i = sum_{j<=i} (0.5 + (i-j)) dt^2 u_j = dt^2 (0.5 S1_i + sum_{j<i} S1_j)
template <int NT>
static __device__ __noinline__ void prims_from_controls(const double *u, double *vth, double *vom, int H, int nj, double dt) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const double dt2 = dt * dt;
#pragma unroll 1
  for (int k = warp; k < nj; k += NT / 32) {
    double carry1 = 0.0, carry2 = 0.0;
#pragma unroll 1
    for (int base = 0; base < H; base += 64) {
      const int i0 = base + 2 * lane, i1 = i0 + 1;
      const double a0 = i0 < H ? u[i0 * nj + k] : 0.0, a1 = i1 < H ? u[i1 * nj + k] : 0.0;
      const double pr = a0 + a1;
      double inc = pr;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const double t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
      }
      const double s0 = carry1 + ((inc - pr) + a0), s1 = carry1 + inc;  // S1 at i0, i1
      const double rr = s0 + s1;
      double inc2 = rr;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const double t = __shfl_up_sync(0xffffffffu, inc2, o);
        if (lane >= o) inc2 += t;
      }
      const double t0 = carry2 + (inc2 - rr), t1 = t0 + s0;  // sum_{j<i} S1_j at i0, i1
      if (i0 < H) {
        vth[i0 * nj + k] = dt2 * (0.5 * s0 + t0);
        vom[i0 * nj + k] = dt * s0;
      }
      if (i1 < H) {
        vth[i1 * nj + k] = dt2 * (0.5 * s1 + t1);
        vom[i1 * nj + k] = dt * s1;
      }
      carry1 = __shfl_sync(0xffffffffu, s1, 31);
      carry2 += __shfl_sync(0xffffffffu, inc2, 31);
    }
  }
}

template <int NT>
static __device__ __noinline__ void qp_refresh_cached(const QpView &s, const QpDims &P, int q) {
  const int n = P.n;
#pragma unroll 1
  for (int c = threadIdx.x; c < n; c += NT) {
    double acc = 0.0;
#pragma unroll 4
    for (int w = 0; w < q; ++w) acc += s.lam[w] * s.zc[(size_t)s.zslot[w] * n + c];
    s.v[2 * n + c] = s.v0s[2 * n + c] - acc;
  }
  __syncthreads();
  prims_from_controls<NT>(s.v + 2 * n, s.v, s.v + n, P.H, P.nj, P.dt);
  __syncthreads();
}

// e_cid' y for y = P z given as (yth | yom | z)
template <bool LIM = false>
static __device__ __forceinline__ double row_dot_prims(int cid, const double *yth, const double *yom, const double *z,
                                                       const QpDims &P, const double *ocoef) {
  if (cid < P.OH) {
    const double *c = ocoef + (size_t)cid * P.nj, *y = yth + wp_of(cid, P.H) * P.nj;
    double acc = 0.0;
#pragma unroll 1
    for (int k = 0; k < P.nj; ++k) acc += c[k] * y[k];
    return acc;
  }
  const int e = cid - P.OH, pr = e >> 1;
  const double val = pr < P.n ? yom[pr] : ((LIM && pr >= 2 * P.n) ? yth[pr - 2 * P.n] : z[pr - P.n]);
  return (e & 1) ? -val : val;
}

// candidate p: z_p = QQ^-1 c_p' into the candidate slot (one pass over <= nj rows of G), y_p = P z_p by prefix sums, then
// sigma = c_p QQ^-1 c_p' = e_p'y_p and g_w = c_w QQ^-1 c_p' = e_w'y_p for every member
template <int NT, bool LIM = false>
static __device__ __noinline__ double qp_candidate_cached(const QpView &s, const QpDims &P, int p, int q) {
  const int tid = threadIdx.x, n = P.n;
  const Desc dp = decode<LIM>(p, P, s.ocoef);
  double *zp = s.zc + (size_t)s.zslot[q] * n;
  const double *__restrict__ Gu = P.G + (size_t)dp.row0 * P.np + 2 * n;  // control block of the candidate's primitive rows
#pragma unroll 1
  for (int c = tid; c < n; c += NT) {
    double acc = 0.0;
    if (dp.nterm == 1) {
      acc = dp.coef * Gu[c];
    } else {
#pragma unroll 1
      for (int k = 0; k < dp.nterm; ++k) acc += dp.cv[k] * Gu[(size_t)k * P.np + c];
    }
    zp[c] = acc;
  }
  __syncthreads();
  prims_from_controls<NT>(zp, s.yp, s.yp + n, P.H, P.nj, P.dt);
  __syncthreads();
#pragma unroll 1
  for (int w = tid; w <= q; w += NT) {
    const double val = row_dot_prims<LIM>(w < q ? s.act[w] : p, s.yp, s.yp + n, zp, P, s.ocoef);
    if (w < q)
      s.g[w] = val;
    else
      s.red[40] = val;
  }
  __syncthreads();
  return s.red[40];
}

// Phase A of every QP: if two CONSECUTIVE obstacle rows have (almost) opposite coefficient vectors -- the gradient flips
// where the reference passes the obstacle -- they ask for opposite displacements one step apart, and with the velocity /
// control rows that pair alone is, in 96 % of the infeasible linearisations (measured on the headline batch), already
// infeasible.  The dual method finds that certificate in ~4 steps when it only sees those rows, but wanders for up to
// hundreds of steps when it always takes the globally most violated row.  So all other obstacle rows are masked
// (inact = 2) first: "infeasible" for a subset of the rows is infeasible for all of them; otherwise qp_solve unmasks and
// simply continues (its working set stays a valid dual active-set state).
template <int NT>
__device__ __forceinline__ int qp_mask_antiparallel(const QpView &s, const QpDims &P) {
  // returns the number of masking levels set: 0 none; 2: level A1 = the most anti-parallel pair only, level A2 = every
  // pair with cos < -0.9 (inact = 2), then all rows (inact = 3)
  const int tid = threadIdx.x, OH = P.OH, H = P.H, nj = P.nj;
  double best = 0.0;
  int bidx = -1;
#pragma unroll 1
  for (int cid = tid; cid < OH; cid += NT) {
    if (wp_of(cid, H) == H - 1) continue;  // the pair (cid, cid+1) must belong to the same obstacle
    const double *a = s.ocoef + (size_t)cid * nj, *b = a + nj;
    double ab = 0.0, aa = 0.0, bb = 0.0;
#pragma unroll 1
    for (int k = 0; k < nj; ++k) {
      ab += a[k] * b[k];
      aa += a[k] * a[k];
      bb += b[k] * b[k];
    }
    if (ab < 0.0 && ab * ab > 0.81 * aa * bb) {  // cos < -0.9
      const double cs = ab / sqrt(aa * bb);
      if (bidx < 0 || cs < best) {
        best = cs;
        bidx = cid;
      }
    }
  }
  block_argmin<NT>(best, bidx, s.red);
  if (bidx < 0) return 0;
#pragma unroll 1
  for (int cid = tid; cid < OH; cid += NT) s.inact[cid] = 3;
  __syncthreads();
#pragma unroll 1
  for (int cid = tid; cid < OH; cid += NT) {
    if (wp_of(cid, H) == H - 1) continue;
    const double *a = s.ocoef + (size_t)cid * nj, *b = a + nj;
    double ab = 0.0, aa = 0.0, bb = 0.0;
#pragma unroll 1
    for (int k = 0; k < nj; ++k) {
      ab += a[k] * b[k];
      aa += a[k] * a[k];
      bb += b[k] * b[k];
    }
    if (ab < 0.0 && ab * ab > 0.81 * aa * bb) {
      s.inact[cid] = 2;
      s.inact[cid + 1] = 2;
    }
  }
  __syncthreads();
  if (tid == 0) {
    s.inact[bidx] = 0;
    s.inact[bidx + 1] = 0;
  }
  __syncthreads();
  return 2;
}

// Polish: the working-set inverse M has been rank-1 updated many times; one step of iterative refinement on
// S_W lambda = b (S_W = C_W QQ^-1 C_W' re-read from G, b = violations at u0) removes the accumulated drift
// (measured: 7e-10 -> 3e-13 in u).
template <int NT, int NJ, bool LIM = false>
static __device__ __noinline__ void qp_polish(const QpView &s, const QpDims &P, int q, const double *M, int ldm) {
  const int tid = threadIdx.x;
  const int nch = NT / q > 0 ? NT / q : 1;  // chunks of columns per row, fixed summation order
  if (q <= NT) {
    const int w = tid % q, ch = tid / q;
    if (ch < nch) {
      double acc = 0.0;
#pragma unroll 1
      for (int c = ch; c < q; c += nch) acc += gram<LIM>(s.act[w], s.act[c], P, s.ocoef) * s.lam[c];
      s.pscr[ch * q + w] = acc;
    }
    __syncthreads();
    if (tid < q) {
      double acc = 0.0;
#pragma unroll 1
      for (int ch2 = 0; ch2 < nch; ++ch2) acc += s.pscr[ch2 * q + tid];
      s.g[tid] = -slack_at<NJ, LIM>(s.act[tid], P, s, s.v0s) - acc;
    }
  } else {
#pragma unroll 1
    for (int w = tid; w < q; w += NT) {
      double acc = 0.0;
#pragma unroll 1
      for (int c = 0; c < q; ++c) acc += gram<LIM>(s.act[w], s.act[c], P, s.ocoef) * s.lam[c];
      s.g[w] = -slack_at<NJ, LIM>(s.act[w], P, s, s.v0s) - acc;
    }
  }
  __syncthreads();
#pragma unroll 1
  for (int w = tid; w < q; w += NT) {
    double acc = 0.0;
#pragma unroll 4
    for (int c = 0; c < q; ++c) acc += M[w + (size_t)ldm * c] * s.g[c];
    s.r[w] = acc;
  }
  __syncthreads();
#pragma unroll 1
  for (int w = tid; w < q; w += NT) s.lam[w] += s.r[w];
  __syncthreads();
}

// Re-factorisation of the working set (G-based tiers): the inverse M of S_W = C_W QQ^-1 C_W' is rebuilt from the Gram operator
// instead of trusted after many rank-1 updates.  Rows that depend on the rows before them (remaining pivot below QP_DEP_TOL of
// their own norm) and rows whose multiplier comes out non-positive leave the set, and the factorisation is repeated on the
// smaller set: what remains has independent rows, positive multipliers lambda = S_W^-1 b (b = violation at the unconstrained
// minimiser) and u(lambda) stationary on it -- a valid state of the dual method, from which qp_solve continues.  Called when
// the working-set residual check finds the updated inverse broken (typically a nearly dependent set on an infeasible QP).
// Returns the new size of the working set, or -1 if no consistent set was reached.
template <int NT, int QS, int NJ, bool LIM = false>
static __device__ __noinline__ int qp_refactor(const QpView &s, const QpDims &P, int q0, double cost0, bool &in_smem,
                                               double *fval_new) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int NW = NT / 32;
  if (q0 > NT || q0 > P.ldg) return -1;  // the column scratch (pscr) holds NT entries
  int qc = q0;
  double *A = nullptr;
  int ld = 0;
  for (int pass = 0;; ++pass) {
    A = qc <= QS ? s.Msm : P.Mgl;
    ld = qc <= QS ? QS : P.ldg;
#pragma unroll 1
    for (int idx = tid; idx < qc * qc; idx += NT) {  // S_W, lower triangle
      const int j = idx / qc, i = idx - j * qc;
      if (i >= j) A[i + (size_t)ld * j] = gram<LIM>(s.act[i], s.act[j], P, s.ocoef);
    }
#pragma unroll 1
    for (int i = tid; i < qc; i += NT) s.g[i] = -slack_at<NJ, LIM>(s.act[i], P, s, s.v0s);
    __syncthreads();
#pragma unroll 1
    for (int i = tid; i < qc; i += NT) {
      s.r[i] = A[i + (size_t)ld * i];
      s.toff[i] = 0;  // "left the set" flags (the term lists are rebuilt below)
    }
    __syncthreads();
    // in-place inverse of the symmetric positive definite matrix by sweeping every row (lower triangle only): afterwards
    // A = -(S^-1) on the swept rows; a dependent row is taken out (zero row and column)
#pragma unroll 1
    for (int k = 0; k < qc; ++k) {
      const double pv = A[k + (size_t)ld * k];
      const bool dep = !(pv > QP_DEP_TOL * s.r[k]);
#pragma unroll 1
      for (int i = tid; i < qc; i += NT) s.pscr[i] = dep ? 0.0 : (i >= k ? A[i + (size_t)ld * k] : A[k + (size_t)ld * i]);
      __syncthreads();
      if (dep) {
#pragma unroll 1
        for (int i = tid; i < qc; i += NT) {
          if (i >= k) A[i + (size_t)ld * k] = 0.0;
          else A[k + (size_t)ld * i] = 0.0;
        }
        if (tid == 0) s.toff[k] = 1;
        __syncthreads();
        continue;
      }
      const double ip = 1.0 / pv;
#pragma unroll 1
      for (int j = warp; j < qc; j += NW) {
        if (j == k) continue;
        const double cj = s.pscr[j] * ip;
#pragma unroll 4
        for (int i = j + lane; i < qc; i += 32)
          if (i != k) A[i + (size_t)ld * j] -= s.pscr[i] * cj;
      }
#pragma unroll 1
      for (int i = tid; i < qc; i += NT) {
        if (i > k) A[i + (size_t)ld * k] = s.pscr[i] * ip;
        else if (i < k) A[k + (size_t)ld * i] = s.pscr[i] * ip;
        else A[k + (size_t)ld * k] = -ip;
      }
      __syncthreads();
    }
    int bad = 0;
#pragma unroll 1
    for (int i = tid; i < qc; i += NT) {  // lambda = S^-1 b
      double acc = 0.0;
#pragma unroll 4
      for (int j = 0; j < qc; ++j) acc += (i >= j ? A[i + (size_t)ld * j] : A[j + (size_t)ld * i]) * s.g[j];
      s.lam[i] = -acc;
      if (s.toff[i] || !(-acc > 0.0)) ++bad;
    }
    __syncthreads();
    const int nbad = (int)(block_sum<NT>((double)bad, s.red) + 0.5);
    if (nbad == 0) break;
    if (pass >= 5) return -1;
    if (tid == 0) {  // take the rows out (a few hundred entries at most: one thread, fixed order)
      int o = 0;
      for (int i = 0; i < qc; ++i) {
        if (s.toff[i] || !(s.lam[i] > 0.0)) {
          s.inact[s.act[i]] = 0;
        } else {
          s.act[o++] = s.act[i];
        }
      }
    }
    qc -= nbad;
    __syncthreads();
    if (qc <= 0) {
      qc = 0;
      break;
    }
  }
  // M = S^-1, both triangles
#pragma unroll 1
  for (int j = warp; j < qc; j += NW)
#pragma unroll 1
    for (int i = j + lane; i < qc; i += 32) {
      const double val = -A[i + (size_t)ld * j];
      A[i + (size_t)ld * j] = val;
      A[j + (size_t)ld * i] = val;
    }
  if (tid == 0) {
    int o = 0;
    for (int w = 0; w < qc; ++w) {
      s.toff[w] = o;
      o += (s.act[w] < P.OH) ? P.nj : 1;
    }
    s.toff[qc] = o;
  }
  __syncthreads();
#pragma unroll 1
  for (int w = tid; w < qc; w += NT) {
    const Desc d = decode<LIM>(s.act[w], P, s.ocoef);
    const int t0 = s.toff[w];
    for (int k = 0; k < d.nterm; ++k) {
      s.trow[t0 + k] = d.row0 + k;
      s.tcoef[t0 + k] = d.cv ? d.cv[k] : d.coef;
      s.towner[t0 + k] = w;
    }
  }
  double part = 0.0;
#pragma unroll 1
  for (int w = tid; w < qc; w += NT) part += s.g[w] * s.lam[w];
  *fval_new = cost0 + 0.5 * block_sum<NT>(part, s.red);  // (also orders the writes above)
  in_smem = qc <= QS;
  __syncthreads();
  return qc;
}

// Solves   min 1/2 u'QQ u + ff'u  s.t. the rows described by (s.ocoef, s.orhs, lim, umax)   starting from the
// unconstrained minimiser whose primitives are in s.v0s / s.v.  On return (status 0) s.v holds the primitives of the
// optimum (controls in s.v[2n..3n)), s.lam / s.act / q the multipliers and the working set.
// status: 0 optimal, 2 infeasible, 3 numerical, 4 escalate (step_cap exceeded / working set outgrew QS and !SPILL).
// Must be called by all NT threads of the CTA.  NJ: compile-time joint count (0 = use P.nj).  LIM: with the joint position
// rows (never masked; s.lim holds qmax | qmin | theta0 from index 8).
template <int NT, int QS, bool SPILL, int NJ, int QZ = 0, bool LIM = false>
__device__ __forceinline__ int qp_solve(const QpView &s, const QpDims &P, double cost0, double fupper, bool skip_solve,
                                        int &q_out, int &steps_out, int &qmax_seen, long long *pf, long long &tck,
                                        bool prof, int step_cap = 0x7fffffff, int masked = 0) {
  const int tid = threadIdx.x;
  const int n = P.n, nj = NJ ? NJ : P.nj, H = P.H, OH = P.OH, has_vel = P.has_vel, has_bnd = P.has_bnd;
  double *Mgl = P.Mgl;
  const int ldg = P.ldg;
  constexpr bool CACHED = QZ > 0;
  int q = 0, status = skip_solve ? 0 : -1, steps = 0;
  bool in_smem = true, polished = false;
  int refactors = 0;
  if (CACHED) {
    if (tid <= QZ) s.zslot[tid] = tid;
    __syncthreads();
  }
  double fval = cost0;
  const int max_steps = 20 * (P.m + n) + 100;
  while (status < 0) {
    double *M = (SPILL && !in_smem) ? Mgl : s.Msm;  // column-major, leading dimension ldm
    const int ldm = (SPILL && !in_smem) ? ldg : QS;
    if (q > 0) {
      if (CACHED)
        qp_refresh_cached<NT>(s, P, q);
      else
        qp_refresh<NT, (SPILL ? 32 : 8)>(s, P, q);
    }
    PF_ADD(QPF(1));
    pf[7] += 1;
    // (1) most violated inactive row, normalised by its QQ^-1 norm: minimise -slack^2/sigma over the violated rows
    double best = 0.0;
    int bidx = -1;
#pragma unroll 1
    for (int j = 0; j < OH; j += H)
#pragma unroll 1
      for (int i = tid; i < H; i += NT) {
        const int cid = j + i;
        const double sg = s.onrm[cid];
        if (s.inact[cid] || !(sg > 0.0)) continue;
        const double *c = s.ocoef + (size_t)cid * nj;
        const double *vv = s.v + i * nj;
        double val = 0.0;
#pragma unroll
        for (int k = 0; k < (NJ ? NJ : 1); ++k) val += c[k] * vv[k];
        if (!NJ)
          for (int k = 1; k < nj; ++k) val += c[k] * vv[k];
        const double sl = s.orhs[cid] - val;
        if (sl < -1e-11 * (1.0 + fabs(s.orhs[cid]))) {
          const double key = -(sl * sl) / sg;
          if (key < best || bidx < 0) {
            best = key;
            bidx = cid;
          }
        }
      }
    // omega / control primitives: both signs of a row share its value and its norm
#pragma unroll 1
    for (int e = tid; e < 2 * n; e += NT) {
      const bool is_w = e < n;
      if (is_w ? !has_vel : !has_bnd) continue;
      const double sg = s.gns[n + e];
      if (!(sg > 0.0)) continue;
      const double vv = s.v[n + e];
      const double hi = prim_rhs<NJ>(e, 0, P, s), lo = prim_rhs<NJ>(e, 1, P, s);
      const double up = hi - vv, dn = lo + vv;
      const double sc = is_w ? 0.5 * (hi + lo) : hi;
      const double tol = 1e-11 * (1.0 + sc);
      const int cu = OH + 2 * e;
      if (up < -tol && !s.inact[cu]) {
        const double key = -(up * up) / sg;
        if (key < best || bidx < 0) {
          best = key;
          bidx = cu;
        }
      }
      if (dn < -tol && !s.inact[cu + 1]) {
        const double key = -(dn * dn) / sg;
        if (key < best || bidx < 0) {
          best = key;
          bidx = cu + 1;
        }
      }
    }
    if (LIM) {  // joint position rows: theta primitives, ids after the control rows
#pragma unroll 1
      for (int e = tid; e < n; e += NT) {
        const double sg = s.gns[e];
        if (!(sg > 0.0)) continue;
        const double vv = s.v[e];
        const double hi = prim_rhs<NJ, LIM>(2 * n + e, 0, P, s), lo = prim_rhs<NJ, LIM>(2 * n + e, 1, P, s);
        const double up = hi - vv, dn = lo + vv;
        const int cu = OH + 4 * n + 2 * e;
        if (up < -1e-11 * (1.0 + fabs(hi)) && !s.inact[cu]) {
          const double key = -(up * up) / sg;
          if (key < best || bidx < 0) {
            best = key;
            bidx = cu;
          }
        }
        if (dn < -1e-11 * (1.0 + fabs(lo)) && !s.inact[cu + 1]) {
          const double key = -(dn * dn) / sg;
          if (key < best || bidx < 0) {
            best = key;
            bidx = cu + 1;
          }
        }
      }
    }
    block_argmin<NT>(best, bidx, s.red);
    PF_ADD(QPF(2));
    if (bidx < 0 && masked) {  // this phase is feasible: unmask the next level and carry on with the same working set
      const int lvl = masked == 2 ? 2 : 3;
#pragma unroll 1
      for (int cid = tid; cid < OH; cid += NT)
        if (s.inact[cid] == lvl) s.inact[cid] = 0;
      --masked;
      __syncthreads();
      if (q == 0) {  // v is still v0: scan again without a refresh
        polished = false;
      }
      continue;
    }
    if (bidx < 0) {
      if (q == 0 || polished || (steps <= 6 && q <= 6)) {  // few updates: M is still accurate to ~1e-13
        if (q > 6) {
          // Safety net: every member of the working set must hold with equality at the recovered point.  On a nearly
          // dependent working set (an infeasible QP on which neither the dependence test nor weak duality has fired yet)
          // the rank-1 updated inverse can lose all accuracy; the scan above only looks at inactive rows and would
          // accept the point.  Such a state is reported as numerical breakdown instead of a wrong "optimal".
          double worst = 0.0;
#pragma unroll 1
          for (int w = tid; w < q; w += NT) {
            const int cw = s.act[w];
            const double rhs = cw < OH ? s.orhs[cw] : prim_rhs<NJ, LIM>((cw - OH) >> 1, (cw - OH) & 1, P, s);
            const double res = fabs(slack_at<NJ, LIM>(cw, P, s, s.v)) / (1.0 + fabs(rhs));
            worst = fmax(worst, res);
          }
          int wi = 0;
          worst = -worst;
          block_argmin<NT>(worst, wi, s.red);
          if (-worst > 1e-6) {
            // broken inverse: rebuild it from the Gram operator (twice at most per QP), drop what does not belong to a valid
            // working set, and continue; the cached tiers (small working sets, no term lists) report the breakdown
            int q1 = -1;
            double fnew = fval;
            if (!CACHED && refactors < 2) {
              ++refactors;
              q1 = qp_refactor<NT, QS, NJ, LIM>(s, P, q, cost0, in_smem, &fnew);
              ++steps;
            }
            if (q1 < 0) {
              status = 3;
              break;
            }
            q = q1;
            fval = fnew;
            polished = false;
            if (fval > fupper) {
              status = 2;
              break;
            }
            continue;
          }
        }
        status = 0;
        break;
      }
      qp_polish<NT, NJ, LIM>(s, P, q, M, ldm);
      polished = true;
      continue;  // re-evaluate v from the refined multipliers and scan once more
    }
    polished = false;
    const int p = bidx;
    // sigma = c_p QQ^-1 c_p': one G entry for a primitive row, an nj x nj bilinear form (one load per thread) otherwise
    double sigma;
    if (CACHED) {
      if (q > QZ - 1) {  // no slot left for the candidate's direction: the heavy tier redoes this iteration
        status = 4;
        break;
      }
      sigma = qp_candidate_cached<NT, LIM>(s, P, p, q);
    } else if (p < OH) {
      double part = 0.0;
      if (tid < nj * nj) {
        const int k = tid / nj, l2 = tid - k * nj, r0 = wp_of(p, H) * nj;
        part = s.ocoef[p * nj + k] * s.ocoef[p * nj + l2] * P.G[(size_t)(r0 + k) * P.np + r0 + l2];
      }
      sigma = block_sum<NT>(part, s.red);
    } else if (LIM) {
      const int r0 = decode<LIM>(p, P, s.ocoef).row0;
      sigma = P.G[(size_t)r0 * P.np + r0];
    } else {
      sigma = P.G[(size_t)(n + ((p - OH) >> 1)) * P.np + n + ((p - OH) >> 1)];
    }
    double sp = slack_at<NJ, LIM>(p, P, s, s.v);
    double lam_p = 0.0;
    // (2) bring row p into the working set
    for (;;) {
      if (++steps > max_steps) {
        status = 3;
        break;
      }
      if (steps > step_cap) {  // hand the problem to the heavy tier (k_fused.cu)
        status = 4;
        break;
      }
      // g_w = c_w QQ^-1 c_p' = sum over the member's terms of coef_t * (G[row_t, :] . c_p): one thread per TERM (<= nj
      // independent L2 loads each) instead of one per member (up to nj x nj dependent ones), then a fixed-order sum per member.
      // twgt is free between two refreshes.
      if (!CACHED) {
        const Desc dp = decode<LIM>(p, P, s.ocoef);
        const int T = s.toff[q];
#pragma unroll 1
        for (int t = tid; t < T; t += NT) {
          const double *__restrict__ Gr = P.G + (size_t)s.trow[t] * P.np + dp.row0;
          double acc;
          if (dp.nterm == 1) {
            acc = dp.coef * Gr[0];
          } else {
            acc = 0.0;
#pragma unroll 6
            for (int l2 = 0; l2 < dp.nterm; ++l2) acc += dp.cv[l2] * Gr[l2];
          }
          s.twgt[t] = s.tcoef[t] * acc;
        }
        __syncthreads();
#pragma unroll 1
        for (int w = tid; w < q; w += NT) {
          double acc = 0.0;
#pragma unroll 1
          for (int t = s.toff[w]; t < s.toff[w + 1]; ++t) acc += s.twgt[t];
          s.g[w] = acc;
        }
        __syncthreads();
      }
      // r = Minv g ;  delta = sigma - g'r  (z'n+ in Goldfarb-Idnani's notation) ; t1 = largest dual step keeping lambda >= 0
      double part = 0.0, t1 = INFINITY;
      int l = -1;
      {
        // rows padded to a multiple of 32 so that a warp owns one column chunk; nsp chunks per row, fixed order
        const int qp = (q + 31) & ~31;
        const int nsp = (qp > 0 && NT / qp > 1) ? NT / qp : 1;
        if (nsp > 1) {
          const int ch = tid / qp, w = tid - ch * qp;
          if (ch < nsp && w < q) {
            double acc = 0.0;
#pragma unroll 4
            for (int c = ch; c < q; c += nsp) acc += M[w + (size_t)ldm * c] * s.g[c];
            s.pscr[ch * qp + w] = acc;
          }
          __syncthreads();
        }
#pragma unroll 1
        for (int w = tid; w < q; w += NT) {
          double acc = 0.0;
          if (nsp > 1) {
#pragma unroll 1
            for (int ch = 0; ch < nsp; ++ch) acc += s.pscr[ch * qp + w];
          } else {
#pragma unroll 8
            for (int c = 0; c < q; ++c) acc += M[w + (size_t)ldm * c] * s.g[c];
          }
          s.r[w] = acc;
          part += s.g[w] * acc;
          if (acc > 0.0) {
            const double t = s.lam[w] / acc;
            if (t < t1 || l < 0) {
              t1 = t;
              l = w;
            }
          }
        }
      }
      const double delta = sigma - block_sum<NT>(part, s.red);
      block_argmin<NT>(t1, l, s.red);
      if (l < 0) t1 = INFINITY;
      if (!(delta == delta) || !(sigma == sigma)) {
        status = 3;
        break;
      }
      // Row p is treated as linearly dependent on the working set when its QQ^-1-orthogonal remainder is below
      // 1e-8 of its norm^2: in Gram form delta carries cancellation noise ~eps*cond(S_W)*sigma, and a step of
      // length -sp/delta along such a direction only manufactures astronomically large multipliers.
      const bool dependent = !(delta > QP_DEP_TOL * sigma) || q >= n;
      double t2 = INFINITY;
      if (!dependent) {
        t2 = -sp / delta;
        if (t2 < 0.0) t2 = 0.0;
      }
      if (l < 0 && dependent) {
        status = 2;  // infeasible
        break;
      }
      const bool full = (t2 <= t1);
      const double t = full ? t2 : t1;
      // dual objective (Goldfarb-Idnani: f += t z'n+ (t/2 + u+_{q+1})); weak duality: if it exceeds an upper bound of
      // the primal objective over the box |u| <= MAX_input the QP has no feasible point.
      if (!dependent) {
        fval += t * delta * (0.5 * t + lam_p);
        sp += t * delta;  // slack of p moves by t z'n+
      }
      if (fval > fupper) {
        status = 2;
        break;
      }
#pragma unroll 1
      for (int w = tid; w < q; w += NT) s.lam[w] -= t * s.r[w];
      lam_p += t;
      __syncthreads();
      PF_ADD(QPF(3));
      if (full) {
        if (in_smem && q + 1 > QS) {
          if (!SPILL) {
            status = 4;
            break;
          }
          // spill the inverse to the global slab
#pragma unroll 1
          for (int c = tid >> 5; c < q; c += NT / 32)
#pragma unroll 1
            for (int r = tid & 31; r < q; r += 32) Mgl[r + (size_t)ldg * c] = s.Msm[r + QS * c];
          in_smem = false;
          __syncthreads();
        }
        double *Mw = (SPILL && !in_smem) ? Mgl : s.Msm;
        const int ldw = (SPILL && !in_smem) ? ldg : QS;
        // add p: bordered inverse  [[M + r r'/d, -r/d], [-r'/d, 1/d]]   (one warp per column, lanes along rows)
        const double id = 1.0 / delta;
#pragma unroll 1
        for (int c = tid >> 5; c <= q; c += NT / 32) {
          const double rc = c < q ? s.r[c] * id : 0.0;
#pragma unroll 4
          for (int r = tid & 31; r <= q; r += 32) {
            double val;
            if (r < q && c < q)
              val = Mw[r + (size_t)ldw * c] + s.r[r] * rc;
            else if (r == q && c == q)
              val = id;
            else
              val = -s.r[r < q ? r : c] * id;
            Mw[r + (size_t)ldw * c] = val;
          }
        }
        if (!CACHED) {
          const Desc dp = decode<LIM>(p, P, s.ocoef);
          const int t0 = s.toff[q];
          if (tid < dp.nterm) {
            s.trow[t0 + tid] = dp.row0 + tid;
            s.tcoef[t0 + tid] = dp.cv ? dp.cv[tid] : dp.coef;
            s.towner[t0 + tid] = q;
          }
          if (tid == 0) s.toff[q + 1] = t0 + dp.nterm;
        }
        if (tid == 0) {
          s.act[q] = p;
          s.lam[q] = lam_p;
          s.inact[p] = 1;
        }
        ++q;
        if (q > qmax_seen) qmax_seen = q;
        __syncthreads();
        PF_ADD(QPF(4));
        break;
      }
      // drop working-set member l: M <- M - M(:,l) M(l,:)/M(l,l), then move the last member into slot l
      {
        const int last = q - 1;
        double *col = CACHED ? s.pscr : s.g;  // cached mode keeps g (it only depends on (w, p))
#pragma unroll 1
        for (int w = tid; w < q; w += NT) col[w] = M[w + (size_t)ldm * l];
        __syncthreads();
        const double ip = 1.0 / col[l];
#pragma unroll 1
        for (int c = tid >> 5; c < q; c += NT / 32) {
          const double gc = col[c] * ip;
#pragma unroll 4
          for (int r = tid & 31; r < q; r += 32) M[r + (size_t)ldm * c] -= col[r] * gc;
        }
        __syncthreads();
        if (l != last) {
#pragma unroll 1
          for (int w = tid; w < q; w += NT) M[w + (size_t)ldm * l] = M[w + (size_t)ldm * last];
          __syncthreads();
#pragma unroll 1
          for (int w = tid; w < q; w += NT) M[l + (size_t)ldm * w] = M[last + (size_t)ldm * w];
        }
        if (tid == 0) {
          s.inact[s.act[l]] = 0;
          s.act[l] = s.act[last];
          s.lam[l] = s.lam[last];
          if (CACHED) {
            // member `last` moves to l, the candidate's slot follows the shrinking working set, l's slot becomes free
            s.g[l] = s.g[last];
            const int freed = s.zslot[l];
            s.zslot[l] = s.zslot[last];
            s.zslot[last] = s.zslot[q];
            s.zslot[q] = freed;
          } else {
            int o = 0;  // rebuild the term offsets (drops are rare)
            for (int w = 0; w < last; ++w) {
              s.toff[w] = o;
              o += (s.act[w] < OH) ? nj : 1;
            }
            s.toff[last] = o;
          }
        }
        --q;
        __syncthreads();
        if (!CACHED) {
#pragma unroll 1
          for (int w = tid; w < q; w += NT) {
            const Desc d = decode<LIM>(s.act[w], P, s.ocoef);
            const int t0 = s.toff[w];
            for (int k = 0; k < d.nterm; ++k) {
              s.trow[t0 + k] = d.row0 + k;
              s.tcoef[t0 + k] = d.cv ? d.cv[k] : d.coef;
              s.towner[t0 + k] = w;
            }
          }
          __syncthreads();
        }
        PF_ADD(QPF(4));
      }
    }
  }
  q_out = q;
  steps_out = steps;
  return status;
}

}  // namespace cfs
