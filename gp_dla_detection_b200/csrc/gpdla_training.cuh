// Training set of the GP null model on the device: learn_qso_model.m:36-75 (spectra -> lya_1pzs, centered_rest_fluxes,
// rest_noise_variances, mu) and the statistics of its PCA initialisation, learn_qso_model.m:82-95 (nanstd of the
// centred fluxes, the pairwise covariance that pca(X, 'rows', 'pairwise') decomposes); the multi-DLA model's variant,
// learn_qso_model_meanflux.m, adds the Lyman-series mean-flux correction and fills NaNs by row medians before its PCA.
//   training_set_kernel         one CTA per spectrum: linear interpolation (interp1) onto the rest grid, noisy pixels,
//                               with LYSERIES also the Kim et al. mean-flux correction of flux and noise variance
//   row_nanmedian_fill_kernel   one CTA per row: NaN -> the row's nanmedian (bitonic sort in shared memory)
//   column_partial_kernel       per-column partial sums over fixed row blocks, then column_finish_kernel sums the blocks
//   pairwise_cov_tile_kernel    lower-triangle 64 x 64 tiles of X~0' X~0 on FP64 DMMA, pairwise counts by popc
//   pairwise_cov_finish_kernel  fixed-order sum of the row-split partials, / (n - 1), mirrored to the full P x P
// No value is accumulated with atomics: every sum has one writer and a fixed order, so repeated calls give the same bits.
#pragma once
#include <stdint.h>
#include <math.h>
// dmma_884 (mma.sync m8n8k4 f64) comes from gpdla_kernels.cuh, included first by gpdla_capi.cu

namespace gpdla {

struct TrainingArgs {
  // spectra, padded [N x L_max] (the planes gpdla_process_qsos reads)
  const double* wavelengths;
  const double* flux;
  const double* noise_variance;
  const uint8_t* pixel_mask;
  const int32_t* lengths;
  const double* z_qsos;
  const double* rest;            // rest_wavelengths [P], strictly increasing
  int64_t N, L_max;
  int P;
  double lya_wavelength;         // set_parameters.m:5
  double max_noise_variance;     // set_parameters.m (1^2), set_parameters_multi.m:37 (3^2)
  double* lya_1pzs;              // [N x P]
  double* rest_fluxes;           // [N x P], centred in place afterwards
  double* rest_noise_variances;  // [N x P]
  // mean-flux correction (training_set_kernel<true> only): forest.num_forest_lines members, their wavelengths (A),
  // Kim weights and prev_beta -- the table inference reads from c_forest, filled by the same host helper
  ForestConstants forest;
  double lya_over_wavelength[MAX_LINES];   // lya_wavelength / forest.wavelength[l], increasing in l
  double* lya_absorption;        // [N x P] or nullptr
};

constexpr int TS_THREADS = 256;

// emitted wavelengths, 1 + z_lya, flux, noise variance; the Lyman-series variant also stages the observed wavelengths
__host__ __device__ constexpr size_t training_set_smem_bytes(int64_t L_max, bool lyseries) {
  return (size_t)L_max * (lyseries ? 5 : 4) * sizeof(double);
}

// interp1(x, v, r) on the interval [x_j, x_{j+1}], every operation rounded on its own (no FMA contraction)
__device__ __forceinline__ double lerp_rn(double t, double v0, double v1) {
  return __dadd_rn(v0, __dmul_rn(t, __dsub_rn(v1, v0)));
}

// 1 + z_l = 1 + (lambda - lambda_l) / lambda_l at an observed wavelength, each operation rounded on its own
__device__ __forceinline__ double one_plus_z_rn(double lam, double lambda_l) {
  return __dadd_rn(1.0, __ddiv_rn(__dsub_rn(lam, lambda_l), lambda_l));
}

// LYSERIES = false: learn_qso_model.m:36-69.  LYSERIES = true: learn_qso_model_meanflux.m, the same interpolation and
// noisy-pixel rule, then every kept pixel divided by the Kim et al. absorption exp(-sum_l kim_tau_l (1 + z_l)^prev_beta)
template <bool LYSERIES>
__global__ void __launch_bounds__(TS_THREADS) training_set_kernel(const __grid_constant__ TrainingArgs a) {
  extern __shared__ __align__(16) double ts_smem[];
  const int64_t i = blockIdx.x;
  const int L = (int)max((int64_t)0, min((int64_t)a.lengths[i], a.L_max));
  double* sx = ts_smem;              // emitted_wavelengths
  double* sw = sx + a.L_max;         // 1 + (lambda - lya) / lya
  double* sf = sw + a.L_max;         // flux, NaN where masked
  double* sv = sf + a.L_max;         // noise variance, NaN where masked
  double* sl = sv + a.L_max;         // observed wavelengths (LYSERIES)
  const double opz = __dadd_rn(1.0, a.z_qsos[i]);
  const double lya = a.lya_wavelength;
  const int64_t row = i * a.L_max;
  for (int j = threadIdx.x; j < L; j += TS_THREADS) {          // learn_qso_model.m:40-50
    const double lam = a.wavelengths[row + j];
    const bool m = a.pixel_mask[row + j] != 0;
    sx[j] = __ddiv_rn(lam, opz);
    sw[j] = __dadd_rn(1.0, __ddiv_rn(__dsub_rn(lam, lya), lya));
    sf[j] = m ? __longlong_as_double(0x7ff8000000000000ll) : a.flux[row + j];
    sv[j] = m ? __longlong_as_double(0x7ff8000000000000ll) : a.noise_variance[row + j];
    if (LYSERIES) sl[j] = lam;
  }
  __syncthreads();
  const double qnan = __longlong_as_double(0x7ff8000000000000ll);
  const int64_t out = i * a.P;
  for (int p = threadIdx.x; p < a.P; p += TS_THREADS) {        // :52-64, then the noisy-pixel rule :66-69
    const double r = a.rest[p];
    double oz = qnan, of = qnan, ov = qnan;
    double total = 0.0;                                        // nansum of the forest terms: 0 where nothing is observed
    if (L >= 2 && r >= sx[0] && r <= sx[L - 1]) {
      int lo = 0, hi = L - 1;                                  // largest j with x_j <= r
      while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (sx[mid] <= r) lo = mid; else hi = mid - 1;
      }
      const int j = min(lo, L - 2);
      const double t = __ddiv_rn(__dsub_rn(r, sx[j]), __dsub_rn(sx[j + 1], sx[j]));
      oz = lerp_rn(t, sw[j], sw[j + 1]);
      of = lerp_rn(t, sf[j], sf[j + 1]);
      ov = lerp_rn(t, sv[j], sv[j + 1]);
      if (ov > a.max_noise_variance) { oz = qnan; of = qnan; ov = qnan; }
      else if (LYSERIES) {
        // sum_l kim_tau_l (1 + z_l)^prev_beta in ascending l; a member below Lya counts where 1 + z_l <= 1 + z_qso.  A
        // failing indicator makes the term +0.0, which leaves the sum's bits alone, so its pow is skipped.  Moreover
        // 1 + z_l equals (1 + z_Lya) lya / lambda_l to a few ulp; where that estimate exceeds 1 + z_qso by a relative
        // 1e-12 the indicator fails for certain, and, the estimate growing with l, for every later member too.  So the
        // loop stops there, and most grid points evaluate one to three members exactly instead of all of them.
        const double l0 = sl[j], l1 = sl[j + 1];
        const double opz_safe = opz * (1.0 + 1e-12);
        for (int l = 0; l < a.forest.num_forest_lines; ++l) {
          if (l > 0 && oz * a.lya_over_wavelength[l] > opz_safe) break;
          const double wl = a.forest.wavelength[l];
          const double zl = lerp_rn(t, one_plus_z_rn(l0, wl), one_plus_z_rn(l1, wl));
          if (l == 0 ? !isnan(zl) : zl <= opz)                 // NaN terms are skipped (nansum)
            total = __dadd_rn(total, __dmul_rn(a.forest.kim_tau[l], pow(zl, a.forest.prev_beta)));
        }
      }
    }
    if (LYSERIES) {
      const double absorption = exp(-total);
      of = __ddiv_rn(of, absorption);                          // NaN stays NaN
      ov = __ddiv_rn(ov, __dmul_rn(absorption, absorption));
      if (a.lya_absorption) a.lya_absorption[out + p] = absorption;
    }
    a.lya_1pzs[out + p] = oz;
    a.rest_fluxes[out + p] = of;
    a.rest_noise_variances[out + p] = ov;
  }
}

// ---- column reductions over an [N x P] row-major matrix with NaN = not observed.  Row block b of COL_ROWS rows gives
// one partial per column (summed in row order by one thread), column_finish_kernel adds the blocks in block order.
constexpr int COL_THREADS = 128;
constexpr int COL_ROWS = 256;
enum ColumnMode : int {
  COL_MEAN = 0,      // sum, count                        -> mean = sum / n, count
  COL_CENTRE = 1,    // x -= centre (written back), sum   -> mean of the centred column (count given)
  COL_SQDEV = 2,     // sum (x - centre)^2                -> sqrt(sum / (n - 1))
};

__global__ void __launch_bounds__(COL_THREADS) column_partial_kernel(double* X, int64_t N, int P, int mode,
                                                                      const double* __restrict__ centre,
                                                                      double* __restrict__ psum, int32_t* __restrict__ pcnt) {
  const int c = blockIdx.x * COL_THREADS + threadIdx.x;
  if (c >= P) return;
  const int64_t r0 = (int64_t)blockIdx.y * COL_ROWS, r1 = min(N, r0 + COL_ROWS);
  const double m = (mode == COL_MEAN) ? 0.0 : centre[c];
  double s = 0.0;
  int n = 0;
#pragma unroll 4
  for (int64_t r = r0; r < r1; ++r) {
    double x = X[r * P + c];
    if (mode == COL_CENTRE) { x = x - m; X[r * P + c] = x; }     // NaN stays NaN
    if (!isnan(x)) {
      if (mode == COL_SQDEV) { const double d = x - m; s += d * d; } else { s += x; }
      ++n;
    }
  }
  psum[(int64_t)blockIdx.y * P + c] = s;
  pcnt[(int64_t)blockIdx.y * P + c] = n;
}

__global__ void column_finish_kernel(const double* __restrict__ psum, const int32_t* __restrict__ pcnt, int nblocks, int P,
                                     int mode, double* __restrict__ out, int32_t* __restrict__ count) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= P) return;
  double s = 0.0;
  int n = 0;
  for (int b = 0; b < nblocks; ++b) { s += psum[(int64_t)b * P + c]; n += pcnt[(int64_t)b * P + c]; }
  const double qnan = __longlong_as_double(0x7ff8000000000000ll);
  if (mode == COL_MEAN) { out[c] = n > 0 ? s / n : qnan; if (count) count[c] = n; }
  else if (mode == COL_CENTRE) out[c] = n > 0 ? s / n : qnan;
  else out[c] = n > 1 ? sqrt(s / (n - 1)) : qnan;
}

// ---- row medians: out[r, p] = X[r, p], or nanmedian(X[r, :]) where X[r, p] is NaN; an all-NaN row stays NaN.  One CTA per
// row sorts the row's values as order-preserving integer keys (NaN and the padding up to a power of two last) with a
// bitonic network in shared memory; no atomics, so the result does not depend on scheduling.
constexpr int MED_THREADS = 512;
constexpr int MED_MAX_P = 16384;               // 128 KB of keys

__host__ __device__ inline int median_sort_size(int P) { int s = 1; while (s < P) s <<= 1; return s; }

__device__ __forceinline__ uint64_t median_key(double v) {     // a < b  <=>  key(a) < key(b); -0 sorts before +0
  const uint64_t b = (uint64_t)__double_as_longlong(v);
  return isnan(v) ? ~0ull : (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double median_value(uint64_t k) {
  return __longlong_as_double((long long)((k >> 63) ? (k & 0x7fffffffffffffffull) : ~k));
}

// MATLAB's median of an even count: meanof(a, b) = a + (b - a) / 2, or (a + b) / 2 where sign(a) ~= sign(b) (sign(0) = 0)
// or either is infinite
__device__ __forceinline__ double matlab_meanof(double a, double b) {
  const int sa = (a > 0.0) - (a < 0.0), sb = (b > 0.0) - (b < 0.0);
  if (sa != sb || isinf(a) || isinf(b)) return __ddiv_rn(__dadd_rn(a, b), 2.0);
  return __dadd_rn(a, __ddiv_rn(__dsub_rn(b, a), 2.0));
}

__global__ void __launch_bounds__(MED_THREADS) row_nanmedian_fill_kernel(const double* X, int P, int S, double* out) {
  extern __shared__ __align__(16) uint64_t med_keys[];
  __shared__ int warp_count[MED_THREADS / 32];
  const int64_t row = (int64_t)blockIdx.x * P;
  int n = 0;
  for (int p = threadIdx.x; p < S; p += MED_THREADS) {
    uint64_t k = ~0ull;
    if (p < P) { const double v = X[row + p]; if (!isnan(v)) { k = median_key(v); ++n; } }
    med_keys[p] = k;
  }
  n = __reduce_add_sync(0xffffffffu, n);
  if ((threadIdx.x & 31) == 0) warp_count[threadIdx.x >> 5] = n;
  __syncthreads();
  int count = 0;
#pragma unroll
  for (int w = 0; w < MED_THREADS / 32; ++w) count += warp_count[w];
  double med = __longlong_as_double(0x7ff8000000000000ll);
  if (count > 0 && count < P) {                  // a complete row has nothing to fill, an all-NaN row nothing to fill with
    for (int k = 2; k <= S; k <<= 1)
      for (int j = k >> 1; j > 0; j >>= 1) {
        for (int e = threadIdx.x; e < S / 2; e += MED_THREADS) {
          const int lo = 2 * e - (e & (j - 1)), hi = lo + j;      // the pairs (lo, lo + j) with bit j of lo clear
          const uint64_t a = med_keys[lo], b = med_keys[hi];
          if ((a > b) == ((lo & k) == 0)) { med_keys[lo] = b; med_keys[hi] = a; }
        }
        __syncthreads();
      }
    med = (count & 1) ? median_value(med_keys[count / 2])
                      : matlab_meanof(median_value(med_keys[count / 2 - 1]), median_value(med_keys[count / 2]));
  }
  for (int p = threadIdx.x; p < P; p += MED_THREADS) {
    const double v = X[row + p];
    out[row + p] = isnan(v) ? med : v;
  }
}

// ---- pairwise covariance C_pq = sum_{rows observed in both} X~_rp X~_rq / (n_pq - 1), X~ = X - nanmean(X)
// A CTA owns one lower-triangle tile (ti >= tj) of TILE x TILE outputs and one contiguous split of the rows.  Rows are
// staged CHUNK at a time into shared memory (coalesced along P, NaN -> 0, the column mean subtracted) together with the
// 32-bit observed mask of every staged column; eight warps each accumulate a 32 x 16 block with m8n8k4 DMMA, and count
// n_pq with popc(mask_p & mask_q) per chunk.  The next chunk is loaded into registers while the current one computes.
// 32 x 16 blocks keep a thread at <= 128 registers, so two CTAs (16 warps) share an SM; with 32 x 32 blocks and 4 warps
// a thread needed 255 registers and the kernel ran at 5.9 against 9.2 TFLOP/s now (one B200, 1000 W; DESIGN.md §10).
constexpr int COV_TILE = 64;
constexpr int COV_CHUNK = 32;                  // rows per stage = bits per mask word
constexpr int COV_THREADS = 256;
constexpr int COV_WM = 32, COV_WN = 16;        // warp block: COV_WM / 8 x COV_WN / 8 m8n8 tiles
constexpr int COV_MT = COV_WM / 8, COV_NT = COV_WN / 8;
constexpr int COV_PARTS = COV_THREADS / COV_TILE;            // row parts of a staged chunk: 4 x 8 rows
static_assert((COV_TILE / COV_WM) * (COV_TILE / COV_WN) * 32 == COV_THREADS, "warp blocks tile the output tile");
static_assert(COV_CHUNK / COV_PARTS == 8, "one mask byte per row part");
constexpr int COV_LD = COV_TILE + 4;           // +4 doubles: the fragment loads of a half-warp hit 16 distinct banks
constexpr int COV_RPT = COV_CHUNK * COV_TILE / COV_THREADS;   // rows staged per thread and operand: 8

struct CovArgs {
  const double* X;          // [N x P]
  const double* mean;       // [P] nanmean of X
  int64_t N;
  int P;
  int ntile;                // lower-triangle tiles
  int64_t rows_per_split;   // multiple of COV_CHUNK
  double* psum;             // [nsplit][ntile][TILE * TILE]
  int32_t* pcnt;            // same layout
};

__host__ __device__ inline void cov_tile_coords(int t, int& ti, int& tj) {
  int i = (int)((sqrt(8.0 * t + 1.0) - 1.0) * 0.5);
  while (i * (i + 1) / 2 > t) --i;
  while ((i + 1) * (i + 2) / 2 <= t) ++i;
  ti = i; tj = t - i * (i + 1) / 2;
}

__global__ void __launch_bounds__(COV_THREADS, 2) pairwise_cov_tile_kernel(CovArgs a) {
  __shared__ __align__(16) double sA[COV_CHUNK][COV_LD];
  __shared__ __align__(16) double sB[COV_CHUNK][COV_LD];
  __shared__ uint8_t sM[2][COV_PARTS][COV_TILE];   // [operand][row part][column] observed bits
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int t = blockIdx.x;
  int ti, tj;
  cov_tile_coords(t, ti, tj);
  const int P = a.P;
  // staging role: one column of each operand, rows h * 8 .. h * 8 + 7 of the chunk
  const int c = tid % COV_TILE, h = tid / COV_TILE;
  const int pa = ti * COV_TILE + c, pb = tj * COV_TILE + c;
  const double ma = pa < P ? a.mean[pa] : 0.0, mb = pb < P ? a.mean[pb] : 0.0;
  const int64_t r_begin = (int64_t)blockIdx.y * a.rows_per_split;
  const int64_t r_end = min(a.N, r_begin + a.rows_per_split);
  double ra[COV_RPT], rb[COV_RPT];
  uint32_t bits_a = 0, bits_b = 0;
  auto load = [&](int64_t r0) {
    bits_a = 0; bits_b = 0;
#pragma unroll
    for (int k = 0; k < COV_RPT; ++k) {
      const int64_t r = r0 + h * COV_RPT + k;
      double xa = 0.0, xb = 0.0;
      if (r < r_end) {
        if (pa < P) { const double v = a.X[r * P + pa]; if (!isnan(v)) { xa = v - ma; bits_a |= 1u << k; } }
        if (pb < P) { const double v = a.X[r * P + pb]; if (!isnan(v)) { xb = v - mb; bits_b |= 1u << k; } }
      }
      ra[k] = xa; rb[k] = xb;
    }
  };
  // compute role: warp w owns the 32 x 16 block (wp, wq); m8n8k4 fragments: A[g][tg], B[tg][g], C[g][2 tg + j]
  constexpr int WQ = COV_TILE / COV_WN;
  const int wp = (warp / WQ) * COV_WM, wq = (warp % WQ) * COV_WN;
  const int g = lane >> 2, tg = lane & 3;
  double acc[COV_MT][COV_NT][2];
  int32_t cnt[COV_MT][COV_NT][2];
#pragma unroll
  for (int m = 0; m < COV_MT; ++m)
#pragma unroll
    for (int n = 0; n < COV_NT; ++n) { acc[m][n][0] = acc[m][n][1] = 0.0; cnt[m][n][0] = cnt[m][n][1] = 0; }

  if (r_begin < r_end) load(r_begin);
  for (int64_t r0 = r_begin; r0 < r_end; r0 += COV_CHUNK) {
    __syncthreads();                                     // the previous chunk is consumed
#pragma unroll
    for (int k = 0; k < COV_RPT; ++k) { sA[h * COV_RPT + k][c] = ra[k]; sB[h * COV_RPT + k][c] = rb[k]; }
    sM[0][h][c] = (uint8_t)bits_a; sM[1][h][c] = (uint8_t)bits_b;
    __syncthreads();
    if (r0 + COV_CHUNK < r_end) load(r0 + COV_CHUNK);   // in flight while this chunk computes
#pragma unroll
    for (int ks = 0; ks < COV_CHUNK / 4; ++ks) {
      double af[COV_MT], bf[COV_NT];
#pragma unroll
      for (int m = 0; m < COV_MT; ++m) af[m] = sA[ks * 4 + tg][wp + m * 8 + g];
#pragma unroll
      for (int n = 0; n < COV_NT; ++n) bf[n] = sB[ks * 4 + tg][wq + n * 8 + g];
#pragma unroll
      for (int m = 0; m < COV_MT; ++m)
#pragma unroll
        for (int n = 0; n < COV_NT; ++n) dmma_884(acc[m][n][0], acc[m][n][1], af[m], bf[n]);
    }
    auto word = [&](int op, int col) {
      uint32_t w = 0;
#pragma unroll
      for (int part = 0; part < COV_PARTS; ++part) w |= (uint32_t)sM[op][part][col] << (8 * part);
      return w;
    };
    uint32_t wa[COV_MT], wb[COV_NT][2];
#pragma unroll
    for (int m = 0; m < COV_MT; ++m) wa[m] = word(0, wp + m * 8 + g);
#pragma unroll
    for (int n = 0; n < COV_NT; ++n)
#pragma unroll
      for (int j = 0; j < 2; ++j) wb[n][j] = word(1, wq + n * 8 + 2 * tg + j);
#pragma unroll
    for (int m = 0; m < COV_MT; ++m)
#pragma unroll
      for (int n = 0; n < COV_NT; ++n) { cnt[m][n][0] += __popc(wa[m] & wb[n][0]); cnt[m][n][1] += __popc(wa[m] & wb[n][1]); }
  }
  const int64_t base = ((int64_t)blockIdx.y * a.ntile + t) * (COV_TILE * COV_TILE);
#pragma unroll
  for (int m = 0; m < COV_MT; ++m)
#pragma unroll
    for (int n = 0; n < COV_NT; ++n) {
      const int64_t e = base + (int64_t)(wp + m * 8 + g) * COV_TILE + wq + n * 8 + 2 * tg;
      *reinterpret_cast<double2*>(a.psum + e) = make_double2(acc[m][n][0], acc[m][n][1]);
      *reinterpret_cast<int2*>(a.pcnt + e) = make_int2(cnt[m][n][0], cnt[m][n][1]);
    }
}

// C_pq from the lower-triangle tile holding (max(p, q), min(p, q)): both halves read the same partials in the same order
__global__ void pairwise_cov_finish_kernel(const double* __restrict__ psum, const int32_t* __restrict__ pcnt, int nsplit,
                                           int ntile, int P, double* __restrict__ cov, int32_t* __restrict__ counts) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= (int64_t)P * P) return;
  const int p = (int)(e / P), q = (int)(e % P);
  const int hi = max(p, q), lo = min(p, q);
  const int ti = hi / COV_TILE, tj = lo / COV_TILE;
  const int t = ti * (ti + 1) / 2 + tj;
  const int64_t off = (int64_t)(hi % COV_TILE) * COV_TILE + lo % COV_TILE;
  double s = 0.0;
  int n = 0;
  for (int sp = 0; sp < nsplit; ++sp) {
    const int64_t idx = ((int64_t)sp * ntile + t) * (COV_TILE * COV_TILE) + off;
    s += psum[idx];
    n += pcnt[idx];
  }
  cov[e] = n >= 2 ? s / (n - 1) : __longlong_as_double(0x7ff8000000000000ll);
  counts[e] = n;
}

}  // namespace gpdla
