// Training set of the GP null model on the device: learn_qso_model.m:36-75 (spectra -> lya_1pzs, centered_rest_fluxes,
// rest_noise_variances, mu) and the statistics of its PCA initialisation, learn_qso_model.m:82-95 (nanstd of the
// centred fluxes, the pairwise covariance that pca(X, 'rows', 'pairwise') decomposes).
//   training_set_kernel         one CTA per spectrum: linear interpolation (interp1) onto the rest grid, noisy pixels
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
  double max_noise_variance;     // set_parameters.m (1^2)
  double* lya_1pzs;              // [N x P]
  double* rest_fluxes;           // [N x P], centred in place afterwards
  double* rest_noise_variances;  // [N x P]
};

constexpr int TS_THREADS = 256;

__host__ __device__ constexpr size_t training_set_smem_bytes(int64_t L_max) { return (size_t)L_max * 4 * sizeof(double); }

// interp1(x, v, r) on the interval [x_j, x_{j+1}], every operation rounded on its own (no FMA contraction)
__device__ __forceinline__ double lerp_rn(double t, double v0, double v1) {
  return __dadd_rn(v0, __dmul_rn(t, __dsub_rn(v1, v0)));
}

__global__ void __launch_bounds__(TS_THREADS) training_set_kernel(TrainingArgs a) {
  extern __shared__ __align__(16) double ts_smem[];
  const int64_t i = blockIdx.x;
  const int L = (int)max((int64_t)0, min((int64_t)a.lengths[i], a.L_max));
  double* sx = ts_smem;              // emitted_wavelengths
  double* sw = sx + a.L_max;         // 1 + (lambda - lya) / lya
  double* sf = sw + a.L_max;         // flux, NaN where masked
  double* sv = sf + a.L_max;         // noise variance, NaN where masked
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
  }
  __syncthreads();
  const double qnan = __longlong_as_double(0x7ff8000000000000ll);
  const int64_t out = i * a.P;
  for (int p = threadIdx.x; p < a.P; p += TS_THREADS) {        // :52-64, then the noisy-pixel rule :66-69
    const double r = a.rest[p];
    double oz = qnan, of = qnan, ov = qnan;
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
