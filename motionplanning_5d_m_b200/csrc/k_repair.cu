// k_repair.cu -- the device side of the checked solve (cfs_solve_checked, include/cfs_b200.h), sm_100a, FP64: repair increments of
// the per-waypoint margin offsets from the witnesses of a continuous check, and the round loop's bookkeeping (stable selection of
// the problems to re-solve, gather / scatter of the sub-batch).  The CPU restatement of the increments is tests/repair_oracle.c.
// A translation unit of its own: the check kernels (k_check.cu) share the out-of-line box distance with any caller in their unit,
// and stay exactly as they were compiled without these kernels.
#include "cfs_geom.cuh"
#include "cfs_kernels.cuh"

namespace cfs {

// ---- repair increments of the checked solve (cfs_solve_checked, include/cfs_b200.h) ------------------------------------------
// One thread per selected trajectory walks its H segments in order (deterministic, like k_check_reduce).  Segment k of a HIT
// verdict: witness theta* = path(s_hit) with the operations of k_check, then per obstacle c_j = min_l d_lj(theta*) - m_j (one FK,
// nobs distances; equal to k_check's clearance for the minimum over j).  inc_j = gain (eta - c_j) where c_j < -eta/2, else 0.
// Waypoint i in 1..H gets max(inc of segment i-1, inc of segment i) added to its offset (waypoint 0 is x0 and cannot move).
// sel[t] (t < *count): position of the trajectory in the checked set (x0 / x / u, per-segment verdict / s_hit);
// map[pos] (or identity when map == nullptr): its problem b in margin_off.
template <int NJ>
__global__ void __launch_bounds__(128) k_repair_margins(CheckArgs a, const int *count, const int *sel, const int *map, double gain,
                                                        double *margin_off) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= *count) return;
  const DevTables &tab = *a.tab;
  const int H = a.H, O = a.nobs, pos = sel[t], b = map ? map[pos] : pos;
  const double half_eta = 0.5 * a.eta;
  double prev[CFS_MAX_OBS], cur[CFS_MAX_OBS];
  for (int j = 0; j < O; ++j) prev[j] = 0.0;
  double *off = margin_off + (size_t)b * O * H;
  for (int k = 0; k < H; ++k) {
    const long long it = (long long)pos * H + k;
    for (int j = 0; j < O; ++j) cur[j] = 0.0;
    if (a.verdict[it] == CHK_HIT) {
      const double *p0 = k == 0 ? a.x0 + (long long)pos * 2 * NJ : a.x + ((long long)pos * H + (k - 1)) * 2 * NJ;
      const double *p1 = p0 + NJ, *pu = a.u + it * NJ;
      const double sh = a.s_hit[it];
      double th[NJ];
#pragma unroll
      for (int q = 0; q < NJ; ++q)
        th[q] = __dadd_rn(__dadd_rn(p0[q], __dmul_rn(p1[q], sh)), __dmul_rn(__dmul_rn(__dmul_rn(0.5, sh), sh), pu[q]));
      double dmin[CFS_MAX_OBS];
      for (int j = 0; j < O; ++j) dmin[j] = INFINITY;
      Xf M;
      double p[6];
      int touched = 0;
#pragma unroll
      for (int l = 0; l < NJ; ++l) {
        double sn, cs;
        sincos(th[l] + tab.link[l].th_off, &sn, &cs);
        if (l == 0)
          xf_first(tab.link[0], cs, sn, M);
        else
          xf_step_inplace(M, tab.link[l], cs, sn);
        link_endpoints(M, tab.link[l], tab.base, p);
        for (int j = 0; j < O; ++j) {
          const double d = key_to_dist(link_obs_key(p, tab.obs[j], touched));
          dmin[j] = d < dmin[j] ? d : dmin[j];
        }
      }
      for (int j = 0; j < O; ++j) {
        const double c = __dsub_rn(dmin[j], a.margin_is_D ? tab.obs[j].D : tab.obs[j].eps);
        if (c < -half_eta) cur[j] = __dmul_rn(gain, __dsub_rn(a.eta, c));
      }
    }
    if (k > 0)
      for (int j = 0; j < O; ++j) {
        const double inc = prev[j] > cur[j] ? prev[j] : cur[j];
        off[(size_t)j * H + (k - 1)] = __dadd_rn(off[(size_t)j * H + (k - 1)], inc);
      }
    for (int j = 0; j < O; ++j) prev[j] = cur[j];
  }
  for (int j = 0; j < O; ++j) off[(size_t)j * H + (H - 1)] = __dadd_rn(off[(size_t)j * H + (H - 1)], prev[j]);
}

cudaError_t launch_repair_margins(const CheckArgs &a, int nmax, const int *count, const int *sel, const int *map, double gain,
                                  double *margin_off, cudaStream_t s) {
  if (nmax <= 0) return cudaSuccess;
  const int grid = (nmax + 127) / 128;
  switch (a.nj) {
    case 2: k_repair_margins<2><<<grid, 128, 0, s>>>(a, count, sel, map, gain, margin_off); break;
    case 3: k_repair_margins<3><<<grid, 128, 0, s>>>(a, count, sel, map, gain, margin_off); break;
    case 4: k_repair_margins<4><<<grid, 128, 0, s>>>(a, count, sel, map, gain, margin_off); break;
    case 5: k_repair_margins<5><<<grid, 128, 0, s>>>(a, count, sel, map, gain, margin_off); break;
    case 6: k_repair_margins<6><<<grid, 128, 0, s>>>(a, count, sel, map, gain, margin_off); break;
    default: return cudaErrorInvalidValue;
  }
  return cudaGetLastError();
}

// ---- the round loop's bookkeeping: stable compaction, gather, scatter ---------------------------------------------------------
// flag of position p: mode 0 (after the first solve): verdict[p] == HIT and status low byte < 2; mode 1 (after a re-solve of the
// sub-batch): the candidate was accepted (status low byte < 2) and its verdict is HIT.  One CTA, positions in increasing order:
// sel = the flagged positions, next[t] = map ? map[sel[t]] : sel[t], *count = their number.
__global__ void __launch_bounds__(1024) k_repair_select(int N, const int *verdict, const int *status, const int *map, int *sel,
                                                        int *next, int *count) {
  __shared__ int wsum[32];
  __shared__ int base;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  if (tid == 0) base = 0;
  __syncthreads();
  for (int p0 = 0; p0 < N; p0 += 1024) {
    const int p = p0 + tid;
    const bool f = p < N && verdict[p] == CHK_HIT && (status[p] & 0xFF) < 2;
    const unsigned m = __ballot_sync(0xffffffffu, f);
    if (lane == 0) wsum[wid] = __popc(m);
    __syncthreads();
    int before = base;
    for (int w = 0; w < wid; ++w) before += wsum[w];
    if (f) {
      const int t = before + __popc(m & ((1u << lane) - 1u));
      sel[t] = p;
      next[t] = map ? map[p] : p;
    }
    __syncthreads();
    if (tid == 0)
      for (int w = 0; w < 32; ++w) base += wsum[w];
    __syncthreads();
  }
  if (tid == 0) *count = base;
}

cudaError_t launch_repair_select(int N, const int *verdict, const int *status, const int *map, int *sel, int *next, int *count,
                                 cudaStream_t s) {
  k_repair_select<<<1, 1024, 0, s>>>(N, verdict, status, map, sel, next, count);
  return cudaGetLastError();
}

// rows of length len: dst[t] = src[list[t]] (gather) or dst[list[t]] = src[t] (scatter), for t < count; scatter rows whose
// status low byte (st[t], or nullptr: all) is >= 2 are skipped.  One CTA per row.
__global__ void k_rows_copy(int n_rows, const int *list, const double *src, double *dst, long long len, int scatter, const int *st) {
  const int t = blockIdx.x;
  if (t >= n_rows) return;
  if (st && (st[t] & 0xFF) >= 2) return;
  const long long si = scatter ? t : list[t], di = scatter ? list[t] : t;
  for (long long e = threadIdx.x; e < len; e += blockDim.x) dst[di * len + e] = src[si * len + e];
}
__global__ void k_ints_copy(int n_rows, const int *list, const int *src, int *dst, int scatter, const int *st, int fill) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_rows) return;
  if (st && (st[t] & 0xFF) >= 2) return;
  const int si = scatter ? t : list[t], di = scatter ? list[t] : t;
  dst[di] = fill >= 0 ? fill : src[si];
}

cudaError_t launch_rows_copy(int n_rows, const int *list, const double *src, double *dst, long long len, int scatter, const int *st,
                             cudaStream_t s) {
  if (n_rows <= 0 || len <= 0) return cudaSuccess;
  k_rows_copy<<<n_rows, 128, 0, s>>>(n_rows, list, src, dst, len, scatter, st);
  return cudaGetLastError();
}
cudaError_t launch_ints_copy(int n_rows, const int *list, const int *src, int *dst, int scatter, const int *st, int fill,
                             cudaStream_t s) {
  if (n_rows <= 0) return cudaSuccess;
  k_ints_copy<<<(n_rows + 127) / 128, 128, 0, s>>>(n_rows, list, src, dst, scatter, st, fill);
  return cudaGetLastError();
}

// 1 in *bad if any of the N offsets is negative or not finite (argument check of cfs_solve_batch_margins_device)
__global__ void k_offsets_bad(long long N, const double *off, int *bad) {
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < N; e += (long long)gridDim.x * blockDim.x) {
    const double v = off[e];
    if (!(v >= 0.0 && v < INFINITY)) *bad = 1;
  }
}
cudaError_t launch_offsets_bad(long long N, const double *off, int *bad, cudaStream_t s) {
  cudaError_t e = cudaMemsetAsync(bad, 0, sizeof(int), s);
  if (e != cudaSuccess || N <= 0) return e;
  long long g = (N + 255) / 256;
  k_offsets_bad<<<(int)(g < 1024 ? g : 1024), 256, 0, s>>>(N, off, bad);
  return cudaGetLastError();
}

}  // namespace cfs
