// Population statistics of the single-DLA catalogue (the additive sums behind CDDF_analysis/calc_cddf.py: f(N_HI, X),
// dN/dX, Omega_DLA) from the device-resident sample log-likelihoods (Bird, Garnett & Ho 2017).
//   stats_class_kernel        per sample: its log-N class (the intervals between the union of the log-N bin edges and
//                             the DLA threshold) and an order-preserving key of its offset
//   stats_rank_kernel         per sample: its rank under (class, offset, index), by counting; perm[rank] = sample
//   stats_gather_kernel       samples in rank order (offset, N), rank[sample], and the first position of every class
//   dla_stats_kernel<STAGED>  one CTA per quasar: the normalised sample posterior, then for every (z bin, class) cell a
//                             fixed-order range sum; writes the quasar's row of cell values in the layout of the sums
//   column_partial_kernel     (gpdla_training.cuh) per-column sums over fixed 256-row blocks of those rows, then
//   stats_finish_kernel       adds the blocks, in block order, into the caller's sums vector
// Within a class the samples are sorted by offset, and z = min_z + (max_z - min_z) * offset is monotone in the offset
// (IEEE multiply and add are monotone), so every (z bin, class) cell is one contiguous range, found by binary search on
// the computed z.  No atomics: repeated calls give the same bits.
#pragma once
#include <stdint.h>
#include <math.h>
// median_key and column_partial_kernel come from gpdla_training.cuh, included first by gpdla_capi.cu

namespace gpdla {

constexpr int STAT_MAX_Z = 64;                        // z bins
constexpr int STAT_MAX_NHI = 128;                     // log-N bins
constexpr int STAT_MAX_BOUND = STAT_MAX_NHI + 2;      // class boundaries: the n_nhi + 1 edges and the DLA threshold
constexpr int STAT_THREADS = 256;
constexpr int STAT_RANK_TILE = 1024;
constexpr int STAT_UNROLL = 8;                        // row loads in flight per thread in the first pass

// sums layout, float64, n_z z bins x n_nhi log-N bins:
//   counts[n_z][n_nhi], counts_var[n_z][n_nhi], dla[n_z], dla_var[n_z], nhi[n_z], nhi_var[n_z], path[n_z], num_quasars
__host__ __device__ constexpr int64_t stats_width(int n_z, int n_nhi) { return 2 * (int64_t)n_z * n_nhi + 5 * n_z + 1; }

struct StatsClassArgs {
  const double* offset;
  const double* log_nhi;
  int64_t S;
  int nbound;                                // m class boundaries, ascending; class k = [bound[k-1], bound[k])
  double bound[STAT_MAX_BOUND];
  int32_t* cls;                              // [S] 0..m: the number of boundaries <= log N (NaN: 0, counts nowhere)
  uint64_t* key;                             // [S] median_key(offset)
};

__global__ void stats_class_kernel(const __grid_constant__ StatsClassArgs a) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= a.S) return;
  const double v = a.log_nhi[j];
  int c = 0;
  for (int k = 0; k < a.nbound; ++k) c += (a.bound[k] <= v);
  a.cls[j] = c;
  a.key[j] = median_key(a.offset[j]);
}

// rank of sample j = #{i : (cls_i, key_i, i) < (cls_j, key_j, j)}: S^2 comparisons, a few microseconds at S = 10^4
__global__ void __launch_bounds__(STAT_THREADS) stats_rank_kernel(const int32_t* __restrict__ cls,
                                                                  const uint64_t* __restrict__ key, int64_t S,
                                                                  int32_t* __restrict__ perm) {
  __shared__ int32_t s_cls[STAT_RANK_TILE];
  __shared__ uint64_t s_key[STAT_RANK_TILE];
  const int64_t j = (int64_t)blockIdx.x * STAT_THREADS + threadIdx.x;
  const int cj = j < S ? cls[j] : 0;
  const uint64_t kj = j < S ? key[j] : 0;
  int64_t r = 0;
  for (int64_t t0 = 0; t0 < S; t0 += STAT_RANK_TILE) {
    __syncthreads();
    for (int t = threadIdx.x; t < STAT_RANK_TILE; t += STAT_THREADS) {
      const int64_t i = t0 + t;
      s_cls[t] = i < S ? cls[i] : INT32_MAX;
      s_key[t] = i < S ? key[i] : ~0ull;
    }
    __syncthreads();
    const int n = (int)min((int64_t)STAT_RANK_TILE, S - t0);
    for (int t = 0; t < n; ++t) {
      const int ci = s_cls[t];
      const uint64_t ki = s_key[t];
      r += (ci < cj) || (ci == cj && (ki < kj || (ki == kj && t0 + t < j)));
    }
  }
  if (j < S) perm[r] = (int32_t)j;
}

// position r: the sample of rank r; class_start[k] = first position of class >= k, k = 0..nbound + 1
__global__ void stats_gather_kernel(const int32_t* __restrict__ perm, const int32_t* __restrict__ cls,
                                    const double* __restrict__ offset, const double* __restrict__ nhi, int64_t S,
                                    int nbound, double* __restrict__ sorted_offset, double* __restrict__ sorted_nhi,
                                    int32_t* __restrict__ rank, int32_t* __restrict__ class_start) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r < S) {
    const int32_t j = perm[r];
    sorted_offset[r] = offset[j];
    sorted_nhi[r] = nhi[j];
    rank[j] = (int32_t)r;
    const int c = cls[j], cprev = r > 0 ? cls[perm[r - 1]] : -1;
    for (int k = cprev + 1; k <= c; ++k) class_start[k] = (int32_t)r;   // classes cprev+1..c start here
    if (r == S - 1)
      for (int k = c + 1; k <= nbound + 1; ++k) class_start[k] = (int32_t)S;
  }
}

struct StatsArgs {
  const double* ll;                          // [Q x S] sample_log_likelihoods_dla
  const double* p_dlas;
  const double* min_z_dlas;
  const double* max_z_dlas;
  const uint8_t* select;                     // nullable
  int64_t S;
  int64_t q0;                                // first quasar of this chunk
  const double* sorted_offset;               // [S] in class-then-offset order
  const double* sorted_nhi;
  const int32_t* perm;                       // position -> sample
  const int32_t* rank;                       // sample -> position
  const int32_t* class_start;                // [nbound + 2]
  int n_z, n_nhi, nbound;
  int64_t W;                                 // stats_width(n_z, n_nhi)
  double z_edges[STAT_MAX_Z + 1];
  int16_t nhi_class0[STAT_MAX_NHI];          // log-N bin c = classes [nhi_class0[c], nhi_class1[c]) (1-based classes)
  int16_t nhi_class1[STAT_MAX_NHI];
  int dla_class0;                            // classes >= dla_class0 are DLAs (log N >= dla_log_nhi_min)
  double omega_m, omega_l, x_coef;           // X(z) = x_coef sqrt(omega_m (1+z)^3 + omega_l), x_coef = 2 / (3 omega_m)
  double* rows;                              // [chunk x W]
};

// absorption distance of flat LambdaCDM without radiation, dX/dz = (1+z)^2 H0 / H(z); every operation rounded on its own
__device__ __forceinline__ double absorption_distance(double z, double om, double ol, double coef) {
  const double a = __dadd_rn(1.0, z);
  return __dmul_rn(coef, sqrt(__dadd_rn(__dmul_rn(om, __dmul_rn(__dmul_rn(a, a), a)), ol)));
}

__device__ __forceinline__ double stats_block_sum(double v, double* red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double s = 0.0;
#pragma unroll
  for (int w = 0; w < STAT_THREADS / 32; ++w) s += red[w];     // every thread adds the warps in the same order
  return s;
}

__host__ __device__ inline size_t stats_smem_bytes(bool staged, int64_t S, int n_z, int nbound) {
  const size_t pos = ((size_t)(n_z + 1) * nbound * sizeof(int32_t) + 15) / 16 * 16;
  return (staged ? (size_t)S * sizeof(double) : 0) + pos + (size_t)nbound * 3 * sizeof(double);
}

// One CTA per quasar.  STAGED: the row is staged in shared memory in class-then-offset order and turned into exp(ll - m)
// in place; otherwise (S too large) every pass reads the row from global memory through perm.
template <bool STAGED>
__global__ void __launch_bounds__(STAT_THREADS) dla_stats_kernel(const __grid_constant__ StatsArgs a) {
  extern __shared__ __align__(16) double st_smem[];
  __shared__ double red[STAT_THREADS / 32];
  __shared__ int s_nan;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t q = a.q0 + blockIdx.x;
  const int64_t S = a.S;
  const int m = a.nbound;
  double* row = a.rows + (int64_t)blockIdx.x * a.W;
  double* sw = st_smem;                                        // [S] (STAGED)
  int32_t* pos = reinterpret_cast<int32_t*>(st_smem + (STAGED ? S : 0));            // [(n_z + 1) x m]
  double* cell = st_smem + (STAGED ? S : 0) + ((size_t)(a.n_z + 1) * m * 4 + 15) / 16 * 2;   // [m x 3]
  const double* ll = a.ll + q * S;

  const double p = a.p_dlas[q], zlo = a.min_z_dlas[q], zhi = a.max_z_dlas[q];
  const bool selected = a.select ? a.select[q] != 0 : true;
  bool ok = selected && isfinite(p) && zhi > zlo;
  double mx = -INFINITY;
  if (ok) {                                                    // max over the row; any NaN makes the LSE NaN
    int nan = 0;
    for (int64_t j0 = tid; j0 < S; j0 += STAT_THREADS * STAT_UNROLL) {   // STAT_UNROLL loads in flight per thread
      double v[STAT_UNROLL];
      int32_t r[STAT_UNROLL];
#pragma unroll
      for (int u = 0; u < STAT_UNROLL; ++u) {
        const int64_t j = j0 + u * STAT_THREADS;
        v[u] = j < S ? ll[j] : -INFINITY;
        if (STAGED) r[u] = j < S ? a.rank[j] : 0;
      }
#pragma unroll
      for (int u = 0; u < STAT_UNROLL; ++u) {
        if (STAGED && j0 + u * STAT_THREADS < S) sw[r[u]] = v[u];
        nan |= isnan(v[u]);
        mx = fmax(mx, v[u]);
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    nan = __any_sync(0xffffffffu, nan);
    if (tid == 0) s_nan = 0;
    __syncthreads();
    if (lane == 0) { red[warp] = mx; if (nan) s_nan = 1; }   // benign: every writer stores 1
    __syncthreads();
    mx = red[0];
#pragma unroll
    for (int w = 1; w < STAT_THREADS / 32; ++w) mx = fmax(mx, red[w]);
    ok = !s_nan && isfinite(mx);                               // then sum exp(ll - mx) lies in [1, S]: the LSE is finite
  }
  if (!ok) {                                                   // contributes nothing, not even path or a count
    for (int64_t c = tid; c < a.W; c += STAT_THREADS) row[c] = 0.0;
    return;
  }
  double tot = 0.0;
#pragma unroll 1
  for (int64_t k = tid; k < S; k += STAT_THREADS) {
    const double w = exp((STAGED ? sw[k] : ll[a.perm[k]]) - mx);
    if (STAGED) sw[k] = w;
    tot += w;
  }
  tot = stats_block_sum(tot, red);
  // pos[e * m + k] = first position of class k + 1 whose z is not below z_edges[e]
  for (int idx = tid; idx < (a.n_z + 1) * m; idx += STAT_THREADS) {
    const int e = idx / m, k = idx - e * m;
    int lo = a.class_start[k + 1], hi = a.class_start[k + 2];
    const double edge = a.z_edges[e], span = __dsub_rn(zhi, zlo);
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (__dadd_rn(zlo, __dmul_rn(span, a.sorted_offset[mid])) < edge) lo = mid + 1; else hi = mid;
    }
    pos[idx] = lo;
  }
  __syncthreads();
  const double scale = p / tot;
  const int64_t nzn = (int64_t)a.n_z * a.n_nhi;
  for (int b = 0; b < a.n_z; ++b) {
    for (int k = warp; k < m; k += STAT_THREADS / 32) {       // one warp per (b, class) cell
      const int r0 = pos[b * m + k], r1 = pos[(b + 1) * m + k];
      const bool dla = k + 1 >= a.dla_class0;
      double s0 = 0.0, s1 = 0.0, s2 = 0.0;
#pragma unroll 1                                               // unrolled, the FP64 exp spills
      for (int r = r0 + lane; r < r1; r += 32) {
        const double w = STAGED ? sw[r] : exp(ll[a.perm[r]] - mx);
        s0 += w;
        if (dla) { const double N = a.sorted_nhi[r], wn = w * N; s1 += wn; s2 += wn * N; }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        s0 += __shfl_xor_sync(0xffffffffu, s0, o);
        s1 += __shfl_xor_sync(0xffffffffu, s1, o);
        s2 += __shfl_xor_sync(0xffffffffu, s2, o);
      }
      if (lane == 0) { cell[3 * k] = s0; cell[3 * k + 1] = s1; cell[3 * k + 2] = s2; }
    }
    __syncthreads();
    for (int c = tid; c < a.n_nhi; c += STAT_THREADS) {
      double s = 0.0;
      for (int k = a.nhi_class0[c]; k < a.nhi_class1[c]; ++k) s += cell[3 * (k - 1)];
      const double qv = scale * s;
      row[b * a.n_nhi + c] = qv;
      row[nzn + b * a.n_nhi + c] = qv * (1.0 - qv);
    }
    if (tid == STAT_THREADS - 1) {
      double d = 0.0, e = 0.0, e2 = 0.0;
      for (int k = a.dla_class0; k <= m; ++k) { d += cell[3 * (k - 1)]; e += cell[3 * (k - 1) + 1]; e2 += cell[3 * (k - 1) + 2]; }
      d *= scale; e *= scale; e2 *= scale;
      double* tail = row + 2 * nzn;
      tail[b] = d;
      tail[a.n_z + b] = d * (1.0 - d);
      tail[2 * a.n_z + b] = e;
      tail[3 * a.n_z + b] = e2 - e * e;
      const double xa = absorption_distance(fmax(a.z_edges[b], zlo), a.omega_m, a.omega_l, a.x_coef);
      const double xb = absorption_distance(fmin(a.z_edges[b + 1], zhi), a.omega_m, a.omega_l, a.x_coef);
      tail[4 * a.n_z + b] = fmax(0.0, xb - xa);
    }
    __syncthreads();                                           // cell is reused by the next z bin
  }
  if (tid == 0) row[a.W - 1] = 1.0;
}

// sums[c] += partial[0][c] + partial[1][c] + ..., left to right in block order
__global__ void stats_finish_kernel(const double* __restrict__ psum, int nblocks, int64_t W, double* __restrict__ sums) {
  const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= W) return;
  double s = sums[c];
  for (int b = 0; b < nblocks; ++b) s += psum[(int64_t)b * W + c];
  sums[c] = s;
}

// ---- the multi-DLA model (Ho et al. 2021): sample i of level j (1-based) places j absorbers, slot 0 at sample i and
// slot t at partners[t - 1][i].  A quasar's count X of a cell is then 0..J, and the row holds its exact mixture mean
// and variance.  With v_j(i) = p_j w_ji and g_t(i) = sum_{j > t} v_j(i), E[X] = sum_i sum_t g_t a_t and
// E[X^2] = E[X] + 2 sum_i sum_{t < t'} g_t' a_t a_t' (a_t: slot t lies in the cell; slot t' exists wherever t' does).
//   multi_dla_stats_kernel    one CTA per quasar: per-level log-sum-exp and the partner bounds check in one pass over
//                             the rows (multi_level_lse, shared with gpdla_posteriors.cuh), then every warp takes 32 samples at a time, merges each sample's slots by
//                             cell in registers, and adds them into a warp-private accumulator: lanes sharing a cell
//                             (__match_any_sync) are summed in lane order by the lowest one.  The warps' accumulators
//                             are added in warp order.  No atomics; the order depends only on the launch shape.
constexpr int MSTAT_MAX_DLAS = 4;

struct MultiStatsArgs {
  const double* ll;                          // [Q x J x S] sample_log_likelihoods_dla
  const int32_t* partners;                   // [Q x (J-1) x S] base_sample_inds, 0-based; nullptr when J == 1
  const double* model_posteriors;            // [Q x (2 + J)]: no DLA, sub-DLA, 1..J DLAs
  const double* min_z_dlas;
  const double* max_z_dlas;
  const uint8_t* select;                     // nullable
  int64_t S;
  int64_t q0;                                // first quasar of this chunk
  int J;
  const double* offset;                      // [S] offset_samples
  const double* nhi;                         // [S] nhi_samples
  const int32_t* cls;                        // [S] log-N class (stats_class_kernel)
  int n_z, n_nhi;
  int64_t W;                                 // stats_width(n_z, n_nhi)
  double z_edges[STAT_MAX_Z + 1];
  int16_t class_bin[STAT_MAX_BOUND + 1];     // log-N bin of each class, -1 outside every bin
  int dla_class0;                            // classes >= dla_class0 are DLAs
  double omega_m, omega_l, x_coef;
  double* rows;                              // [chunk x W]
};

// accumulator doubles per warp: (E[X], E[X^2]) per (z bin, log-N bin) cell, then (d, d2, e, e2) per z bin
__host__ __device__ inline int mstats_acc_width(int n_z, int n_nhi) { return 2 * n_z * n_nhi + 4 * n_z; }
__host__ __device__ inline size_t mstats_smem_bytes(int nwarps, int n_z, int n_nhi) {
  return (size_t)nwarps * (mstats_acc_width(n_z, n_nhi) + 32 * 4 + MSTAT_MAX_DLAS * 2) * sizeof(double);
}

// running log-sum-exp (m, s = sum exp(v - m)); NaN and -inf carry no weight, s == 0 means nothing seen
__device__ __forceinline__ void lse_push(double& m, double& s, double v) {
  if (!(v > -INFINITY)) return;
  if (v > m) { s = s * exp(m - v) + 1.0; m = v; } else s += exp(v - m);
}
__device__ __forceinline__ void lse_merge(double& m, double& s, double m2, double s2) {   // commutative
  if (s2 == 0.0) return;
  if (s == 0.0) { m = m2; s = s2; return; }
  const double mm = fmax(m, m2);
  s = s * exp(m - mm) + s2 * exp(m2 - mm);
  m = mm;
}

// Pass 1 of both multi-DLA reductions (this file and gpdla_posteriors.cuh), one read of the J rows [J x S] of a quasar:
// every thread of the CTA gets each level's log-sum-exp (m, s) over the levels in `use` (s == 0: nothing seen), merged
// in a fixed order, and the returned mask has bit t set when partner row t < nrows holds an index outside [0, S).
// Shared memory: red [nwarps x MSTAT_MAX_DLAS x 2] doubles, s_bad [nwarps] ints.
__device__ __forceinline__ int multi_level_lse(const double* __restrict__ ll, const int32_t* __restrict__ part, int64_t S,
                                               const bool use[MSTAT_MAX_DLAS], int nrows, double* red, int* s_bad,
                                               double m[MSTAT_MAX_DLAS], double s[MSTAT_MAX_DLAS]) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = blockDim.x >> 5;
#pragma unroll
  for (int j = 0; j < MSTAT_MAX_DLAS; ++j) { m[j] = -INFINITY; s[j] = 0.0; }
  int bad = 0;
  for (int64_t i = tid; i < S; i += blockDim.x) {
    double v[MSTAT_MAX_DLAS];
    int32_t k[MSTAT_MAX_DLAS - 1];
#pragma unroll
    for (int j = 0; j < MSTAT_MAX_DLAS; ++j) v[j] = use[j] ? ll[j * S + i] : NAN;
#pragma unroll
    for (int t = 0; t < MSTAT_MAX_DLAS - 1; ++t) k[t] = t < nrows ? part[t * S + i] : 0;
#pragma unroll
    for (int j = 0; j < MSTAT_MAX_DLAS; ++j) lse_push(m[j], s[j], v[j]);
#pragma unroll
    for (int t = 0; t < MSTAT_MAX_DLAS - 1; ++t) bad |= ((k[t] < 0) | (k[t] >= S)) << t;
  }
#pragma unroll
  for (int j = 0; j < MSTAT_MAX_DLAS; ++j)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
      lse_merge(m[j], s[j], __shfl_xor_sync(0xffffffffu, m[j], o), __shfl_xor_sync(0xffffffffu, s[j], o));
  bad = __reduce_or_sync(0xffffffffu, bad);
  if (lane == 0) {
    s_bad[warp] = bad;
#pragma unroll
    for (int j = 0; j < MSTAT_MAX_DLAS; ++j) { red[(warp * MSTAT_MAX_DLAS + j) * 2] = m[j]; red[(warp * MSTAT_MAX_DLAS + j) * 2 + 1] = s[j]; }
  }
  __syncthreads();
  bad = 0;
#pragma unroll
  for (int j = 0; j < MSTAT_MAX_DLAS; ++j) {                   // every thread adds the warps in the same order
    m[j] = red[j * 2]; s[j] = red[j * 2 + 1];
    for (int w = 1; w < nw; ++w) lse_merge(m[j], s[j], red[(w * MSTAT_MAX_DLAS + j) * 2], red[(w * MSTAT_MAX_DLAS + j) * 2 + 1]);
  }
  for (int w = 0; w < nw; ++w) bad |= s_bad[w];
  return bad;
}

__global__ void __launch_bounds__(STAT_THREADS) multi_dla_stats_kernel(const __grid_constant__ MultiStatsArgs a) {
  extern __shared__ __align__(16) double ms_smem[];
  __shared__ int s_bad[STAT_THREADS / 32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = blockDim.x >> 5;
  const int64_t q = a.q0 + blockIdx.x, S = a.S;
  const int J = a.J, nzn = a.n_z * a.n_nhi, A = mstats_acc_width(a.n_z, a.n_nhi);
  double* acc = ms_smem;                                       // [nw][A]
  double* stage = acc + (size_t)nw * A;                        // [nw][32][4]
  double* red = stage + nw * 128;                              // [nw][MSTAT_MAX_DLAS][2]
  double* row = a.rows + (int64_t)blockIdx.x * a.W;
  const double* ll = a.ll + q * J * S;
  const int32_t* part = a.partners ? a.partners + q * (J - 1) * S : nullptr;
  const double* mp = a.model_posteriors + q * (J + 2);
  const double zlo = a.min_z_dlas[q], zhi = a.max_z_dlas[q];
  bool ok = (a.select ? a.select[q] != 0 : true) && zhi > zlo;
  for (int c = 0; c < J + 2; ++c) ok = ok && isfinite(mp[c]);
  double p[MSTAT_MAX_DLAS];
  bool use[MSTAT_MAX_DLAS];
  int jmax = 0;                                                // levels 1..jmax can contribute; partner rows < jmax - 1
#pragma unroll
  for (int j = 0; j < MSTAT_MAX_DLAS; ++j) {
    p[j] = (ok && j < J) ? mp[2 + j] : 0.0;
    use[j] = p[j] > 0.0;
    if (use[j]) jmax = j + 1;
  }
  double m[MSTAT_MAX_DLAS], s[MSTAT_MAX_DLAS];
  if (ok) {                                                    // ok is the same for the whole CTA
    const int bad = multi_level_lse(ll, part, S, use, jmax - 1, red, s_bad, m, s);   // pass 1: per-level LSE, partner bounds
#pragma unroll
    for (int j = 0; j < MSTAT_MAX_DLAS; ++j)
      if (p[j] > 0.0 && !isfinite(m[j])) ok = false;           // then s lies in [1, S]
    ok = ok && !bad;
  }
  if (!ok) {                                                   // contributes nothing, not even path or a count
    for (int64_t c = tid; c < a.W; c += blockDim.x) row[c] = 0.0;
    return;
  }
  double sc[MSTAT_MAX_DLAS];
#pragma unroll
  for (int j = 0; j < MSTAT_MAX_DLAS; ++j) sc[j] = p[j] > 0.0 ? p[j] / s[j] : 0.0;
  double* accw = acc + (size_t)warp * A;
  double* st = stage + warp * 128;
  for (int e = lane; e < A; e += 32) accw[e] = 0.0;
  __syncwarp();
  const double span = __dsub_rn(zhi, zlo);
  for (int64_t i0 = (int64_t)warp * 32; i0 < S; i0 += (int64_t)nw * 32) {   // pass 2: 32 samples per warp step
    const int64_t i = i0 + lane;
    double g[MSTAT_MAX_DLAS];                                  // g[t] = sum over levels j >= t (0-based) of p_j w_ji
#pragma unroll
    for (int j = 0; j < MSTAT_MAX_DLAS; ++j) {
      const double x = (i < S && sc[j] > 0.0) ? ll[j * S + i] : NAN;
      g[j] = x == x ? exp(x - m[j]) * sc[j] : 0.0;
    }
#pragma unroll
    for (int t = MSTAT_MAX_DLAS - 2; t >= 0; --t) g[t] += g[t + 1];
    // this sample's slots merged by cell: item u is keyed by the first slot that lands in its cell
    int xk[MSTAT_MAX_DLAS], xn[MSTAT_MAX_DLAS], dk[MSTAT_MAX_DLAS], dn[MSTAT_MAX_DLAS];
    double xm[MSTAT_MAX_DLAS], xs[MSTAT_MAX_DLAS], dm[MSTAT_MAX_DLAS], ds[MSTAT_MAX_DLAS], de[MSTAT_MAX_DLAS],
        de2[MSTAT_MAX_DLAS], dN[MSTAT_MAX_DLAS];
#pragma unroll
    for (int t = 0; t < MSTAT_MAX_DLAS; ++t) {
      xk[t] = dk[t] = -1; xn[t] = dn[t] = 0;
      xm[t] = xs[t] = dm[t] = ds[t] = de[t] = de2[t] = dN[t] = 0.0;
      if (!(g[t] > 0.0)) continue;                             // g is non-increasing in t: no pair needs this slot
      const int64_t k = t == 0 ? i : (int64_t)part[(t - 1) * S + i];   // in [0, S): checked in pass 1
      const double z = __dadd_rn(zlo, __dmul_rn(span, a.offset[k]));
      int lo = 0, hi = a.n_z + 1;                              // number of edges <= z
      while (lo < hi) { const int mid = (lo + hi) >> 1; if (a.z_edges[mid] <= z) lo = mid + 1; else hi = mid; }
      const int b = lo - 1;
      if (b < 0 || b >= a.n_z) continue;
      const int cl = a.cls[k], c = a.class_bin[cl];
      const double gt = g[t];
      if (c >= 0) {
        const int key = b * a.n_nhi + c;
        bool merged = false;
#pragma unroll
        for (int u = 0; u < t; ++u)
          if (!merged && xk[u] == key) {                       // pairs with the xn[u] earlier slots: 2 g_t each
            xm[u] += gt; xs[u] += gt * (double)(1 + 2 * xn[u]); xn[u] += 1; merged = true;
          }
        if (!merged) { xk[t] = key; xm[t] = gt; xs[t] = gt; xn[t] = 1; }
      }
      if (cl >= a.dla_class0) {
        const double N = a.nhi[k], gN = gt * N;
        bool merged = false;
#pragma unroll
        for (int u = 0; u < t; ++u)
          if (!merged && dk[u] == b) {
            dm[u] += gt; ds[u] += gt * (double)(1 + 2 * dn[u]);
            de[u] += gN; de2[u] += gN * N + 2.0 * gN * dN[u];
            dN[u] += N; dn[u] += 1; merged = true;
          }
        if (!merged) { dk[t] = b; dm[t] = gt; ds[t] = gt; de[t] = gN; de2[t] = gN * N; dN[t] = N; dn[t] = 1; }
      }
    }
    // into the warp's accumulator: the lowest lane of each cell adds its lanes in lane order
#pragma unroll
    for (int u = 0; u < MSTAT_MAX_DLAS; ++u) {
      if (u >= J) break;
      unsigned grp = __match_any_sync(0xffffffffu, xk[u]);
      st[lane * 4] = xm[u]; st[lane * 4 + 1] = xs[u];
      __syncwarp();
      if (xk[u] >= 0 && lane == __ffs(grp) - 1) {
        double s0 = 0.0, s1 = 0.0;
        for (unsigned r = grp; r; r &= r - 1) { const int l = __ffs(r) - 1; s0 += st[l * 4]; s1 += st[l * 4 + 1]; }
        accw[2 * xk[u]] += s0; accw[2 * xk[u] + 1] += s1;
      }
      __syncwarp();
      grp = __match_any_sync(0xffffffffu, dk[u]);
      st[lane * 4] = dm[u]; st[lane * 4 + 1] = ds[u]; st[lane * 4 + 2] = de[u]; st[lane * 4 + 3] = de2[u];
      __syncwarp();
      if (dk[u] >= 0 && lane == __ffs(grp) - 1) {
        double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
        for (unsigned r = grp; r; r &= r - 1) {
          const int l = __ffs(r) - 1;
          s0 += st[l * 4]; s1 += st[l * 4 + 1]; s2 += st[l * 4 + 2]; s3 += st[l * 4 + 3];
        }
        double* d = accw + 2 * nzn + 4 * dk[u];
        d[0] += s0; d[1] += s1; d[2] += s2; d[3] += s3;
      }
      __syncwarp();
    }
  }
  __syncthreads();
  for (int e = tid; e < A; e += blockDim.x) {                  // the warps in warp order, into warp 0's copy
    double t = acc[e];
    for (int w = 1; w < nw; ++w) t += acc[(size_t)w * A + e];
    acc[e] = t;
  }
  __syncthreads();
  for (int c = tid; c < nzn; c += blockDim.x) {
    const double mean = acc[2 * c];
    row[c] = mean;
    row[nzn + c] = acc[2 * c + 1] - mean * mean;
  }
  double* tail = row + 2 * nzn;
  for (int b = tid; b < a.n_z; b += blockDim.x) {
    const double* d = acc + 2 * nzn + 4 * b;
    tail[b] = d[0];
    tail[a.n_z + b] = d[1] - d[0] * d[0];
    tail[2 * a.n_z + b] = d[2];
    tail[3 * a.n_z + b] = d[3] - d[2] * d[2];
    const double xa = absorption_distance(fmax(a.z_edges[b], zlo), a.omega_m, a.omega_l, a.x_coef);
    const double xb = absorption_distance(fmin(a.z_edges[b + 1], zhi), a.omega_m, a.omega_l, a.x_coef);
    tail[4 * a.n_z + b] = fmax(0.0, xb - xa);
  }
  if (tid == 0) row[a.W - 1] = 1.0;
}

}  // namespace gpdla
