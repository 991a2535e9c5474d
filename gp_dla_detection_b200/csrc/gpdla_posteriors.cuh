// Per-quasar summaries of the absorber posterior over the DLA samples (the samples are prior draws, so the normalised
// w_i = exp(ll_i - max ll) is the DLA-model posterior over the sample set, process_qsos.m:203-210).
//   posterior_chunk_kernel       per call: the position in offset order of every log-N-ordered sample, laid out so
//                                that thread t of a CTA reads its chunk [t C, t C + C) of the log-N order coalesced
//   dla_posterior_kernel<STAGED> one CTA per quasar: Kish's effective sample size, two-pass central moments of z_DLA
//                                and log N_HI, the posterior mass at log N >= a threshold, and lower inverse-CDF
//                                quantiles of z and log N from fixed-order block scans of the weights
//   multi_dla_posterior_kernel   one CTA per quasar of the multi-DLA model: per level j, its effective sample size and
//                                the moments of the absorber of rank r (ascending z, then log N, then slot), r < j
//   multi_dla_posterior_quantile_kernel<STAGED>   per level j and rank r < j: the mass at log N >= a threshold and
//                                lower inverse-CDF quantiles of z and log N, from fixed-point histograms over the
//                                positions of the absorbers' source samples in the two orders
// No per-quasar sort: z_i = min_z + (max_z - min_z) * offset_i is monotone in offset_i (see gpdla_statistics.cuh) and
// log N_i does not depend on the quasar, so one permutation by offset and one by log N (stats_rank_kernel with one
// class) order every row, and every multi-DLA absorber is one of the samples.  No float atomics: repeated calls give
// the same bits.
#pragma once
#include <stdint.h>
#include <math.h>
// STAT_THREADS, STAT_UNROLL, stats_block_sum, multi_level_lse and MSTAT_MAX_DLAS come from gpdla_statistics.cuh

namespace gpdla {

constexpr int POST_MAX_P = 16;                        // quantile probabilities per call
constexpr int POST_THREADS = STAT_THREADS;
constexpr int MPOST_UNROLL = 4;                      // samples per thread whose gathers are in flight together

// record: ess, z_mean, z_sd, log_nhi_mean, log_nhi_sd, z_log_nhi_cov, mass_above_threshold, z_q[P], log_nhi_q[P]
__host__ __device__ constexpr int64_t posterior_width(int P) { return 7 + 2 * (int64_t)P; }
// record: level-major, level j = ess_j, then (z_mean, z_sd, log_nhi_mean, log_nhi_sd) of the absorbers of rank 0..j-1
__host__ __device__ constexpr int64_t multi_posterior_width(int J) { return J + 2 * (int64_t)J * (J + 1); }
// samples per thread in a scan; odd, so that a warp's strided shared-memory reads hit distinct banks
__host__ __device__ inline int64_t posterior_chunk(int64_t S) { return ((S + POST_THREADS - 1) / POST_THREADS) | 1; }

// n_chunk[i * POST_THREADS + t] = offset-order position of the sample at log-N position t C + i, -1 past S
__global__ void posterior_chunk_kernel(const int32_t* __restrict__ n_perm, const int32_t* __restrict__ z_rank,
                                       int64_t S, int64_t C, int32_t* __restrict__ n_chunk) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= C * POST_THREADS) return;
  const int64_t r = (e % POST_THREADS) * C + e / POST_THREADS;
  n_chunk[e] = r < S ? z_rank[n_perm[r]] : -1;
}

struct PostArgs {
  const double* ll;                          // [Q x S] sample_log_likelihoods_dla
  const double* min_z_dlas;
  const double* max_z_dlas;
  int64_t S, C;                              // C = posterior_chunk(S)
  const double* z_offset;                    // [S] offset_samples in offset order
  const double* z_lnhi;                      // [S] log_nhi_samples in offset order
  const int32_t* z_perm;                     // offset position -> sample
  const int32_t* z_rank;                     // sample -> offset position
  const double* n_lnhi;                      // [S] log_nhi_samples in log-N order
  const int32_t* n_chunk;                    // [C x POST_THREADS] (posterior_chunk_kernel)
  int P;
  double prob[POST_MAX_P];
  double threshold;
  double* out;                               // [Q x posterior_width(P)]
};

// The lower inverse CDF of the weights wt(i) of this thread's chunk [t C, t C + n) of one order: s_pos[p] = the first
// position whose cumulative weight reaches prob[p] * total, total the cumulative weight at the last position.  The
// cumulative weight at chunk position i is E_t + L_i, L_i the chunk's running sum and E_t the exclusive sum of the
// chunk totals (warp scan, then the warps in order); it is monotone inside a chunk, so the first position lies in the
// first chunk whose end reaches the target, and only that chunk's thread walks it again.
template <class Weight>
__device__ __forceinline__ void posterior_quantiles(int64_t S, int64_t C, int P, const double* prob, Weight wt,
                                                    int* s_pos) {
  __shared__ double s_warp[POST_THREADS / 32];
  __shared__ double s_total;
  __shared__ int s_cand[POST_MAX_P][POST_THREADS / 32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t k0 = (int64_t)tid * C;
  const int n = (int)max((int64_t)0, min(C, S - k0));
  double c = 0.0;
#pragma unroll 4
  for (int i = 0; i < n; ++i) c += wt(i);
  double incl = c;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const double y = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += y;
  }
  double excl = __shfl_up_sync(0xffffffffu, incl, 1);
  if (lane == 0) excl = 0.0;
  if (lane == 31) s_warp[warp] = incl;
  __syncthreads();
  double base = 0.0;
  for (int w = 0; w < warp; ++w) base += s_warp[w];
  const double E = base + excl, end = E + c;
  if (n > 0 && k0 + n == S) s_total = end;                     // the chunk holding position S - 1
  __syncthreads();
  const double total = s_total;
  for (int p = 0; p < P; ++p) {
    const unsigned b = __ballot_sync(0xffffffffu, n > 0 && end >= prob[p] * total);
    if (lane == 0) s_cand[p][warp] = b ? warp * 32 + __ffs(b) - 1 : INT32_MAX;
  }
  __syncthreads();
  unsigned own = 0;
  for (int p = 0; p < P; ++p) {
    int f = INT32_MAX;
#pragma unroll
    for (int w = 0; w < POST_THREADS / 32; ++w) f = min(f, s_cand[p][w]);
    if (f == tid) own |= 1u << p;
  }
  c = 0.0;
  if (own) {
#pragma unroll 4
    for (int i = 0; i < n; ++i) {                              // the same sums as above, so the end is reached
      c += wt(i);
      const double cum = E + c;
      for (int p = 0; p < P; ++p)
        if (((own >> p) & 1u) && cum >= prob[p] * total) { s_pos[p] = (int)(k0 + i); own &= ~(1u << p); }
    }
  }
  __syncthreads();
}

// One CTA per quasar.  STAGED: the row is staged in shared memory in offset order and turned into weights in place;
// otherwise (S too large) every pass reads it from global memory through z_perm.
template <bool STAGED>
__global__ void __launch_bounds__(POST_THREADS) dla_posterior_kernel(const __grid_constant__ PostArgs a) {
  extern __shared__ __align__(16) double ps_smem[];
  __shared__ double red[POST_THREADS / 32];
  __shared__ int s_pos[POST_MAX_P];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t q = blockIdx.x, S = a.S, C = a.C;
  const int P = a.P;
  double* rec = a.out + q * posterior_width(P);
  double* sw = ps_smem;                                        // [S] (STAGED)
  const double* ll = a.ll + q * S;
  const double zlo = a.min_z_dlas[q], zhi = a.max_z_dlas[q];
  bool ok = zhi > zlo;
  double mx = -INFINITY;
  if (ok) {                                                    // pass 1: the maximum; NaN and -inf carry no weight
    for (int64_t j0 = tid; j0 < S; j0 += POST_THREADS * STAT_UNROLL) {
      double v[STAT_UNROLL];
      int32_t r[STAT_UNROLL];
#pragma unroll
      for (int u = 0; u < STAT_UNROLL; ++u) {
        const int64_t j = j0 + u * POST_THREADS;
        v[u] = j < S ? ll[j] : -INFINITY;
        if (STAGED) r[u] = j < S ? a.z_rank[j] : 0;
      }
#pragma unroll
      for (int u = 0; u < STAT_UNROLL; ++u) {
        if (STAGED && j0 + u * POST_THREADS < S) sw[r[u]] = v[u];
        mx = fmax(mx, v[u]);                                   // fmax drops NaN
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if (lane == 0) red[warp] = mx;
    __syncthreads();
    mx = red[0];
#pragma unroll
    for (int w = 1; w < POST_THREADS / 32; ++w) mx = fmax(mx, red[w]);
    ok = isfinite(mx);                                         // red is next written after stats_block_sum's barrier
  }
  if (!ok) {                                                   // no finite weight or an empty z range
    for (int c = tid; c < posterior_width(P); c += POST_THREADS) rec[c] = NAN;
    return;
  }
  const double span = __dsub_rn(zhi, zlo);
  auto weight = [&](double v) { return v > -INFINITY ? exp(v - mx) : 0.0; };
  auto z_at = [&](int64_t k) { return __dadd_rn(zlo, __dmul_rn(span, a.z_offset[k])); };   // as map_z_dlas
  double s0 = 0.0, s1 = 0.0, sz = 0.0, sn = 0.0, st = 0.0;    // pass 2: weights, block sums
#pragma unroll 4                                               // the sample arrays come from L2: keep loads in flight
  for (int64_t k = tid; k < S; k += POST_THREADS) {
    const double w = weight(STAGED ? sw[k] : ll[a.z_perm[k]]);
    if (STAGED) sw[k] = w;
    const double z = z_at(k), n = a.z_lnhi[k];
    s0 += w; s1 += w * w; sz += w * z; sn += w * n;
    if (n >= a.threshold) st += w;
  }
  s0 = stats_block_sum(s0, red); s1 = stats_block_sum(s1, red); sz = stats_block_sum(sz, red);
  sn = stats_block_sum(sn, red); st = stats_block_sum(st, red);
  const double zm = sz / s0, nm = sn / s0;
  double czz = 0.0, cnn = 0.0, czn = 0.0;                      // pass 3: central sums
#pragma unroll 4
  for (int64_t k = tid; k < S; k += POST_THREADS) {
    const double w = STAGED ? sw[k] : weight(ll[a.z_perm[k]]);
    const double dz = z_at(k) - zm, dn = a.z_lnhi[k] - nm;
    czz += w * dz * dz; cnn += w * dn * dn; czn += w * dz * dn;
  }
  czz = stats_block_sum(czz, red); cnn = stats_block_sum(cnn, red); czn = stats_block_sum(czn, red);
  if (tid == 0) {
    rec[0] = s0 * s0 / s1;
    rec[1] = zm; rec[2] = sqrt(czz / s0);
    rec[3] = nm; rec[4] = sqrt(cnn / s0);
    rec[5] = czn / s0;
    rec[6] = st / s0;
  }
  const int64_t k0 = (int64_t)tid * C;
  // z: the chunk of offset positions [t C, t C + C)
  posterior_quantiles(S, C, P, a.prob, [&](int i) {
    return STAGED ? sw[k0 + i] : weight(ll[a.z_perm[k0 + i]]);
  }, s_pos);
  if (tid < P) rec[7 + tid] = z_at(s_pos[tid]);
  __syncthreads();                                             // s_pos is reused
  // log N: the chunk of log-N positions, each weight gathered from its offset position
  posterior_quantiles(S, C, P, a.prob, [&](int i) {
    const int zp = a.n_chunk[(int64_t)i * POST_THREADS + tid];
    return zp < 0 ? 0.0 : STAGED ? sw[zp] : weight(ll[a.z_perm[zp]]);
  }, s_pos);
  if (tid < P) rec[7 + P + tid] = a.n_lnhi[s_pos[tid]];
}

// ---- the multi-DLA model: sample i of level j places j absorbers, at i and partners[0..j-2][i]
struct MultiPostArgs {
  const double* ll;                          // [Q x J x S] sample_log_likelihoods_dla
  const int32_t* partners;                   // [Q x (J-1) x S] base_sample_inds, 0-based; nullptr when J == 1
  const double* min_z_dlas;
  const double* max_z_dlas;
  int64_t S;
  int J;
  const double* offset;                      // [S] offset_samples
  const double* log_nhi;                     // [S] log_nhi_samples
  double* out;                               // [Q x multi_posterior_width(J)]
};

// SRC: the source samples ka, kb travel with their slots
template <bool SRC>
__device__ __forceinline__ void slot_exchange(double& za, double& na, int& sa, int& ka, double& zb, double& nb, int& sb,
                                              int& kb) {
  if (za > zb || (za == zb && (na > nb || (na == nb && sa > sb)))) {
    double t = za; za = zb; zb = t;
    t = na; na = nb; nb = t;
    const int u = sa; sa = sb; sb = u;
    if (SRC) { const int v = ka; ka = kb; kb = v; }
  }
}

// the j absorbers of sample i in ascending (z, log N, slot); entries j..3 are +inf.  SRC: src[r] = the sample the
// absorber of rank r comes from (i or a partner), 0 past j
template <bool SRC = false>
__device__ __forceinline__ void sorted_slots(const MultiPostArgs& a, const int32_t* part, int64_t i, int j, double zlo,
                                             double span, double z[MSTAT_MAX_DLAS], double n[MSTAT_MAX_DLAS],
                                             int src[MSTAT_MAX_DLAS] = nullptr) {
  int s[MSTAT_MAX_DLAS], kk[MSTAT_MAX_DLAS];
#pragma unroll
  for (int t = 0; t < MSTAT_MAX_DLAS; ++t) {
    s[t] = t;
    kk[t] = 0;
    z[t] = n[t] = INFINITY;
    if (t < j) {
      const int64_t k = t == 0 ? i : (int64_t)part[(t - 1) * a.S + i];   // in [0, S): checked in pass 1
      kk[t] = (int)k;
      z[t] = __dadd_rn(zlo, __dmul_rn(span, a.offset[k]));
      n[t] = a.log_nhi[k];
    }
  }
  slot_exchange<SRC>(z[0], n[0], s[0], kk[0], z[1], n[1], s[1], kk[1]);
  slot_exchange<SRC>(z[2], n[2], s[2], kk[2], z[3], n[3], s[3], kk[3]);
  slot_exchange<SRC>(z[0], n[0], s[0], kk[0], z[2], n[2], s[2], kk[2]);
  slot_exchange<SRC>(z[1], n[1], s[1], kk[1], z[3], n[3], s[3], kk[3]);
  slot_exchange<SRC>(z[1], n[1], s[1], kk[1], z[2], n[2], s[2], kk[2]);
  if (SRC) {
#pragma unroll
    for (int t = 0; t < MSTAT_MAX_DLAS; ++t) src[t] = kk[t];
  }
}

__global__ void __launch_bounds__(STAT_THREADS) multi_dla_posterior_kernel(const __grid_constant__ MultiPostArgs a) {
  __shared__ double red[STAT_THREADS / 32 * MSTAT_MAX_DLAS * 2];
  __shared__ int s_bad[STAT_THREADS / 32];
  const int tid = threadIdx.x;
  const int64_t q = blockIdx.x, S = a.S;
  const int J = a.J;
  double* rec = a.out + q * multi_posterior_width(J);
  const double* ll = a.ll + q * J * S;
  const int32_t* part = a.partners ? a.partners + q * (J - 1) * S : nullptr;
  const double zlo = a.min_z_dlas[q], zhi = a.max_z_dlas[q];
  if (!(zhi > zlo)) {
    for (int c = tid; c < multi_posterior_width(J); c += STAT_THREADS) rec[c] = NAN;
    return;
  }
  bool use[MSTAT_MAX_DLAS];
#pragma unroll
  for (int j = 0; j < MSTAT_MAX_DLAS; ++j) use[j] = j < J;
  double m[MSTAT_MAX_DLAS], s[MSTAT_MAX_DLAS];
  const int bad = multi_level_lse(ll, part, S, use, J - 1, red, s_bad, m, s);   // pass 1
  const double span = __dsub_rn(zhi, zlo);
  double* lev = rec;
  for (int j = 1; j <= J; ++j) {
    const int L = 1 + 4 * j;
    const double mj = m[j - 1];
    if (!isfinite(mj) || (bad & ((1 << (j - 1)) - 1))) {     // no finite weight, or a partner row outside [0, S)
      for (int c = tid; c < L; c += STAT_THREADS) lev[c] = NAN;
      lev += L;
      continue;
    }
    const double* row = ll + (int64_t)(j - 1) * S;
    // every sample's slots are gathered, weight or not (w = 0 adds 0), so that the loads of a batch overlap
    double s0 = 0.0, s1 = 0.0, sz[MSTAT_MAX_DLAS] = {}, sn[MSTAT_MAX_DLAS] = {};
#pragma unroll MPOST_UNROLL
    for (int64_t i = tid; i < S; i += STAT_THREADS) {          // pass A: sums
      const double v = row[i];
      const double w = v > -INFINITY ? exp(v - mj) : 0.0;
      double z[MSTAT_MAX_DLAS], n[MSTAT_MAX_DLAS];
      sorted_slots(a, part, i, j, zlo, span, z, n);
      s0 += w; s1 += w * w;
#pragma unroll
      for (int r = 0; r < MSTAT_MAX_DLAS; ++r)
        if (r < j) { sz[r] += w * z[r]; sn[r] += w * n[r]; }
    }
    s0 = stats_block_sum(s0, red); s1 = stats_block_sum(s1, red);
    double zm[MSTAT_MAX_DLAS], nm[MSTAT_MAX_DLAS];
#pragma unroll
    for (int r = 0; r < MSTAT_MAX_DLAS; ++r)
      if (r < j) { zm[r] = stats_block_sum(sz[r], red) / s0; nm[r] = stats_block_sum(sn[r], red) / s0; }
    double cz[MSTAT_MAX_DLAS] = {}, cn[MSTAT_MAX_DLAS] = {};
#pragma unroll MPOST_UNROLL
    for (int64_t i = tid; i < S; i += STAT_THREADS) {          // pass B: central sums
      const double v = row[i];
      const double w = v > -INFINITY ? exp(v - mj) : 0.0;
      double z[MSTAT_MAX_DLAS], n[MSTAT_MAX_DLAS];
      sorted_slots(a, part, i, j, zlo, span, z, n);
#pragma unroll
      for (int r = 0; r < MSTAT_MAX_DLAS; ++r)
        if (r < j) {
          const double dz = z[r] - zm[r], dn = n[r] - nm[r];
          cz[r] += w * dz * dz; cn[r] += w * dn * dn;
        }
    }
    double sdz[MSTAT_MAX_DLAS], sdn[MSTAT_MAX_DLAS];
#pragma unroll
    for (int r = 0; r < MSTAT_MAX_DLAS; ++r)
      if (r < j) { sdz[r] = sqrt(stats_block_sum(cz[r], red) / s0); sdn[r] = sqrt(stats_block_sum(cn[r], red) / s0); }
    if (tid == 0) {
      lev[0] = s0 * s0 / s1;
#pragma unroll
      for (int r = 0; r < MSTAT_MAX_DLAS; ++r)
        if (r < j) { lev[1 + 4 * r] = zm[r]; lev[2 + 4 * r] = sdz[r]; lev[3 + 4 * r] = nm[r]; lev[4 + 4 * r] = sdn[r]; }
    }
    lev += L;
  }
}

// ---- credible intervals of every rank of the multi-DLA model.  The rank-r absorber of sample i of level j is a sample
// k = src_r(i) (i or a partner), so its z and log N sit at positions z_rank[k] and n_rank[k] of the two sample orders
// whatever the quasar: its weighted CDF is a histogram over S positions, bin z_rank[k] receiving w_ji, scanned in
// order by posterior_quantiles.  The bins hold sum floor(w 2^F) as uint64, F = 63 - ceil(log2 S): the largest weight
// is exactly 1, so the total lies in [2^F, 2^63], and integer atomics are associative, so the bins, and the record,
// are the same bits on every call whatever the order the threads arrive in.
// record: level-major, then rank; per (level j, rank r < j): mass_above_threshold, z_q[P], log_nhi_q[P]
__host__ __device__ constexpr int64_t multi_quantile_width(int J, int P) {
  return (int64_t)J * (J + 1) / 2 * (1 + 2 * (int64_t)P);
}
__host__ __device__ inline int multi_quantile_bits(int64_t S) {   // F
  int c = 0;
  while (((int64_t)1 << c) < S) ++c;
  return 63 - c;
}
constexpr int MQ_UNROLL = 4;                         // samples per thread whose gathers are in flight together

struct MultiQuantArgs {
  MultiPostArgs m;                           // m.out: [Q x multi_quantile_width(J, P)]
  int64_t Q, C;                              // C = posterior_chunk(S)
  const int32_t* z_rank;                     // sample -> offset position
  const int32_t* n_rank;                     // sample -> log-N position
  const double* z_offset;                    // [S] offset_samples in offset order
  const double* n_lnhi;                      // [S] log_nhi_samples in log-N order
  uint64_t* hist;                            // [gridDim.x x 2 S] per-CTA bins when not STAGED
  int P;
  double prob[POST_MAX_P];
  double threshold;
  double scale;                              // 2^F
};

// A CTA steps over the quasars (STAGED: one each).  Pass 1 is multi_level_lse; then, per level j and rank r < j, one
// pass over the samples fills both histograms (STAGED: in shared memory, otherwise the CTA's global scratch) and the
// float sums of the mass, and two scans read the quantiles.  Lanes of a warp that hit one bin (crowded partners) are
// added by the group's lowest lane, so a bin takes one atomic per warp and sample step.
template <bool STAGED>
__global__ void __launch_bounds__(POST_THREADS) multi_dla_posterior_quantile_kernel(const __grid_constant__ MultiQuantArgs a) {
  extern __shared__ __align__(16) uint64_t mq_smem[];
  __shared__ double red[POST_THREADS / 32 * MSTAT_MAX_DLAS * 2];
  __shared__ int s_bad[POST_THREADS / 32];
  __shared__ uint64_t s_fw[POST_THREADS];
  __shared__ int s_pos[POST_MAX_P];
  __shared__ double s_m[MSTAT_MAX_DLAS];
  const int tid = threadIdx.x, lane = tid & 31;
  const int64_t S = a.m.S, C = a.C;
  const int J = a.m.J, P = a.P, B = 1 + 2 * P;
  const int64_t W = multi_quantile_width(J, P);
  uint64_t* hz = STAGED ? mq_smem : a.hist + (int64_t)blockIdx.x * 2 * S;   // [S] by z position, then [S] by log N
  uint64_t* hn = hz + S;
  uint64_t* fw_warp = s_fw + (tid & ~31);
  bool use[MSTAT_MAX_DLAS];
#pragma unroll
  for (int j = 0; j < MSTAT_MAX_DLAS; ++j) use[j] = j < J;
  auto scan = [&](const uint64_t* h) {                         // one instantiation of posterior_quantiles' statics
    const uint64_t* hk = h + (int64_t)tid * C;
    posterior_quantiles(S, C, P, a.prob, [&](int i) { return (double)(STAGED ? hk[i] : __ldcg(hk + i)); }, s_pos);
  };
  for (int64_t q = blockIdx.x; q < a.Q; q += gridDim.x) {
    __syncthreads();                                           // the previous quasar's reads of red and s_bad are done
    double* rec = a.m.out + q * W;
    const double* ll = a.m.ll + q * J * S;
    const int32_t* part = a.m.partners ? a.m.partners + q * (J - 1) * S : nullptr;
    const double zlo = a.m.min_z_dlas[q], zhi = a.m.max_z_dlas[q];
    if (!(zhi > zlo)) {
      for (int64_t c = tid; c < W; c += POST_THREADS) rec[c] = NAN;
      continue;
    }
    double m[MSTAT_MAX_DLAS], s[MSTAT_MAX_DLAS];
    const int bad = multi_level_lse(ll, part, S, use, J - 1, red, s_bad, m, s);   // pass 1, as the moments kernel
    if (tid < MSTAT_MAX_DLAS) s_m[tid] = tid == 0 ? m[0] : tid == 1 ? m[1] : tid == 2 ? m[2] : m[3];
    __syncthreads();                                           // indexed by level from shared memory, not the stack
    const double span = __dsub_rn(zhi, zlo);
    double* lev = rec;
    for (int j = 1; j <= J; ++j) {
      const double mj = s_m[j - 1];
      if (!isfinite(mj) || (bad & ((1 << (j - 1)) - 1))) {   // no finite weight, or a partner row outside [0, S)
        for (int c = tid; c < j * B; c += POST_THREADS) lev[c] = NAN;
        lev += j * B;
        continue;
      }
      const double* row = ll + (int64_t)(j - 1) * S;
      for (int r = 0; r < j; ++r, lev += B) {
        for (int64_t k = tid; k < 2 * S; k += POST_THREADS) hz[k] = 0;
        __syncthreads();
        double s0 = 0.0, st = 0.0;
        for (int64_t i0 = 0; i0 < S; i0 += POST_THREADS * MQ_UNROLL) {   // block-uniform: whole warps step together
          uint64_t fw[MQ_UNROLL];
          int zb[MQ_UNROLL], nb[MQ_UNROLL];
#pragma unroll
          for (int u = 0; u < MQ_UNROLL; ++u) {
            const int64_t i = i0 + u * POST_THREADS + tid;
            fw[u] = 0; zb[u] = nb[u] = -1;
            const double v = i < S ? row[i] : -INFINITY;
            const double w = v > -INFINITY ? exp(v - mj) : 0.0;
            if (w > 0.0) {
              double z[MSTAT_MAX_DLAS], n[MSTAT_MAX_DLAS];
              int src[MSTAT_MAX_DLAS];
              sorted_slots<true>(a.m, part, i, j, zlo, span, z, n, src);
              int k = 0;
              double nr = 0.0;
#pragma unroll
              for (int t = 0; t < MSTAT_MAX_DLAS; ++t)
                if (t == r) { k = src[t]; nr = n[t]; }
              s0 += w;
              if (nr >= a.threshold) st += w;
              fw[u] = __double2ull_rz(w * a.scale);          // w <= 1, so at most 2^F; exact product, floor
              if (fw[u]) { zb[u] = a.z_rank[k]; nb[u] = a.n_rank[k]; }
            }
          }
#pragma unroll
          for (int u = 0; u < MQ_UNROLL; ++u) {
            fw_warp[lane] = fw[u];
            const unsigned gz = __match_any_sync(0xffffffffu, zb[u]);
            const unsigned gn = __match_any_sync(0xffffffffu, nb[u]);
            __syncwarp();
            if (zb[u] >= 0 && lane == __ffs(gz) - 1) {
              uint64_t t = 0;
              for (unsigned g = gz; g; g &= g - 1) t += fw_warp[__ffs(g) - 1];
              atomicAdd((unsigned long long*)(hz + zb[u]), (unsigned long long)t);
            }
            if (nb[u] >= 0 && lane == __ffs(gn) - 1) {
              uint64_t t = 0;
              for (unsigned g = gn; g; g &= g - 1) t += fw_warp[__ffs(g) - 1];
              atomicAdd((unsigned long long*)(hn + nb[u]), (unsigned long long)t);
            }
            __syncwarp();
          }
        }
        s0 = stats_block_sum(s0, red);                         // its barriers also end the pass's atomics
        st = stats_block_sum(st, red);
        scan(hz);
        if (tid < P) lev[1 + tid] = __dadd_rn(zlo, __dmul_rn(span, a.z_offset[s_pos[tid]]));   // as sorted_slots
        __syncthreads();                                       // s_pos is reused
        scan(hn);
        if (tid < P) lev[1 + P + tid] = a.n_lnhi[s_pos[tid]];
        if (tid == 0) lev[0] = st / s0;
      }
    }
  }
}

}  // namespace gpdla
