// sm_100a kernels of the per-quasar DLA model-selection hot path.
//
//   K0  prepare_quasars_kernel   process_qsos.m:96-181   window/mask, priors, model interpolation,
//                                                        z range, padded grid, Gram operand P
//   K1  voigt_batch_kernel       voigt.c:253-304         stand-alone absorption profiles (API `voigt`)
//   K1+K2+K3 dla_loglik_ws_kernel process_qsos.m:185-199 + log_mvnpdf_low_rank.m:5-34, fused:
//        Voigt profile -> weights -> FP64 DMMA Gram/projection -> Cholesky, log-det, quadratic form
//   K4  evidence_kernel          process_qsos.m:203-233 + generate_ascii_catalog.m:73-80
//
// Reformulation (SURVEY.md 7.2): with a = absorption, d = a^2 omega^2 + v, w = a^2/d, u = a (y - a mu)/d
//   B_s - I = sum_i w_i m_i m_i'   ->  [S x n] . [n x k(k+1)/2]   (operand P, shared by all samples)
//   g_s     = sum_i u_i m_i        ->  [S x n] . [n x k]
//   log p_s = -1/2 ( sum r^2/d - |R'^-1 g|^2 + sum log d + log det B + n log 2pi ),  R'R = B.
#pragma once
#include <stdint.h>
#include "gpdla_math.cuh"

namespace gpdla {

constexpr int KC = 32;            // pixels per K-chunk of the Gram contraction
constexpr int RAWW = 64;          // circular raw-profile buffer width (>= KC + 6, power of two)
constexpr int NTHREADS = 256;     // 8 warps per CTA
constexpr double LOG_2PI = 1.83787706640934534;   // log_mvnpdf_low_rank.m:7

struct QuasarMeta {               // one per quasar, written by K0
  int n_u;                        // pixels inside the modelled window (incl. masked)   process_qsos.m:104-108
  int n;                          // pixels used (window & ~mask)                       process_qsos.m:110
  int nchunks;                    // ceil(n_u / KC)
  int first;                      // index of the first window pixel in the spectrum
  double min_z_dla, max_z_dla;    // process_qsos.m:159-160
  double log_prior_no_dla, log_prior_dla;   // process_qsos.m:128-131
  int prior_num_quasars, prior_num_dlas;    // the counts behind them (multi-DLA priors, ...meanflux.m:190-216)
  double lam_ref;                 // first wavelength of the padded grid: lamh[p] = ln(lam_pad[p] / lam_ref) / h
};

// Lyman-series forest data for the mean-flux suppression of the multi-DLA path
// (multi_dlas/set_parameters_multi.m:76-145, ...meanflux.m:36-37,243-293); filled by the host.
struct ForestConstants {
  double wavelength[MAX_LINES];     // all_transition_wavelengths (Angstrom) = cm value * 1e8
  double tau_ratio[MAX_LINES];      // lambda_l f_l / (lambda_1 f_1)                       ...meanflux.m:255-256
  double kim_tau[MAX_LINES];        // prev_tau_0 f_l / f_lya * lambda_l / lya_wavelength  ...meanflux.m:271-273
  double prev_beta;                 // 3.65
  int num_forest_lines;             // 31
};
__constant__ ForestConstants c_forest;

template <int K>
struct GramShape {
  static constexpr int NPAIR = K * (K + 1) / 2;
  static constexpr int WT = (NPAIR + 7) / 8;     // n8 tiles fed by the W operand
  static constexpr int UT = (K + 7) / 8;         // n8 tiles fed by the U operand
  static constexpr int NT = WT + UT;
  static constexpr int NCOL = NT * 8;
  // row stride of a P chunk in doubles: == 4 (mod 16) makes the DMMA B-fragment loads conflict-free
  static constexpr int BSTR = NCOL + ((4 - NCOL % 16) + 16) % 16;
  static constexpr int CHUNK_DOUBLES = KC * BSTR;
  __host__ __device__ static constexpr int pair_index(int p, int q) { return p * K - p * (p - 1) / 2 + (q - p); }
};

// Column split: ranks whose 8 x NCOL accumulator tile does not fit one warp's registers (k = 40: 864
// columns) are processed by NSPLIT CTAs per sample tile (grid.z), each owning NT / NSPLIT n8 tiles and
// re-evaluating the (comparatively cheap) profile stage; the Cholesky then runs as a separate kernel.
template <int K, int NSPLIT>
struct SplitShape {
  using G = GramShape<K>;
  static_assert(G::NT % NSPLIT == 0, "n8 tiles must divide evenly among the column splits");
  static constexpr int NTL = G::NT / NSPLIT;     // n8 tiles per CTA
  static constexpr int NCOLL = NTL * 8;
  static constexpr int BSTR = NCOLL + ((4 - NCOLL % 16) + 16) % 16;
  static constexpr int CHUNK_DOUBLES = KC * BSTR;
};

constexpr int ASTR = KC + 4;      // row stride of the W/U operand tiles (== 4 mod 16)

// Epilogue staging layout: the symmetric Gram (p <= q < K) and the projected vector (q = K) as one
// augmented upper triangle, entry (p, q) at aug_index(p, q).  stage_index_table<K>() maps an accumulator column
// to that index (-1 for padding columns); filled by the host for every compiled rank.
template <int K>
__host__ __device__ constexpr int aug_index(int p, int q) { return p * (K + 1) - p * (p - 1) / 2 + (q - p); }
// One table per compiled rank (contexts of different rank may share a device).
__constant__ short c_stage_index_10[GramShape<10>::NCOL];
__constant__ short c_stage_index_20[GramShape<20>::NCOL];
__constant__ short c_stage_index_40[GramShape<40>::NCOL];
template <int K> __device__ __forceinline__ const short* stage_index_table();
template <> __device__ __forceinline__ const short* stage_index_table<10>() { return c_stage_index_10; }
template <> __device__ __forceinline__ const short* stage_index_table<20>() { return c_stage_index_20; }
template <> __device__ __forceinline__ const short* stage_index_table<40>() { return c_stage_index_40; }

// ------------------------------------------------------------------------------------------
// small helpers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// 1-D TMA bulk copy global -> shared, completion on an mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void tma_load_1d(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void dmma_884(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ------------------------------------------------------------------------------------------
// K0: per-quasar preparation.  One CTA per quasar.
struct PrepArgs {
  // spectra, padded [Q x L_max]
  const double* wavelengths;
  const double* flux;
  const double* noise_variance;
  const uint8_t* pixel_mask;
  const int32_t* lengths;
  const double* z_qsos;
  int64_t L_max;
  // null model on the rest grid
  const double* rest_wavelengths;
  const double* mu;
  const double* M;          // [n_rest x k] row-major
  const double* log_omega;
  int n_rest, k;
  double c_0, tau_0, beta;
  // prior catalogue
  const double* prior_z_qsos;
  const uint8_t* prior_dla_ind;
  int64_t n_prior;
  // parameters (set_parameters.m)
  double min_lambda, max_lambda, lya_wavelength, lyman_limit, prior_z_qso_increase, min_z_cut, max_z_cut,
      pixel_spacing;
  // outputs
  QuasarMeta* meta;
  double* lam_pad;          // [Q x (NPIX + 8)]
  double* lamh;             // [Q x (NPIX + 8)]  ln(lam_pad / lam_pad[0]) / h: position on the rest-frame table's grid
  double inv_h;             // 1 / (pixel_spacing ln 10)
  double* pix;              // [Q x NPIX x 4]  (y, v, mu, omega2)
  double* Mq;               // [Q x NPIX x k]  interpolated M rows (zero for masked / padding pixels)
  int NPIX;
  int meanflux;             // 1: Lyman-series mean-flux suppression + noise scaling (multi-DLA path)
};

__device__ __forceinline__ double interp_linear(const double* xp, const double* fp, int stride, int j, double x) {
  // numpy.interp / griddedInterpolant('linear') on the bracketing interval j (process_qsos.m:66-71)
  double slope = (fp[(j + 1) * stride] - fp[j * stride]) / (xp[j + 1] - xp[j]);
  return slope * (x - xp[j]) + fp[j * stride];
}

// The null model at one window pixel (observed wavelength w, emitted wavelength rest): process_qsos.m:138-146, and in
// mean-flux mode ...meanflux.m:245-293.  Returns the bracketing rest interval j and
//   mu     interpolated mu, NOT suppressed (mu~ = mu * absorb)
//   om2    omega~^2: interpolated omega^2 times the forest noise scaling and, in mean-flux mode, absorb^2
//   absorb the mean-flux suppression factor s (1 outside mean-flux mode); row c of M~ is interp(M_c) * absorb
// prepare_quasars_kernel and reconstruct_kernel both evaluate the model through this function.
struct PixelModel {
  int j;
  double mu, om2, absorb;
};
__device__ __forceinline__ PixelModel null_model_pixel(const double* __restrict__ rest_wavelengths,
                                                       const double* __restrict__ mu, const double* __restrict__ log_omega,
                                                       int n_rest, double c_0, double tau_0, double beta,
                                                       double lya_wavelength, int meanflux, double w, double rest,
                                                       double z_qso) {
  PixelModel pm;
  const double x0 = rest_wavelengths[0];
  const double inv_dx = (n_rest - 1) / (rest_wavelengths[n_rest - 1] - x0);
  int j = (int)((rest - x0) * inv_dx);
  j = max(0, min(j, n_rest - 2));
  while (j > 0 && rest_wavelengths[j] > rest) --j;
  while (j < n_rest - 2 && rest_wavelengths[j + 1] <= rest) ++j;
  pm.j = j;
  pm.mu = interp_linear(rest_wavelengths, mu, 1, j, rest);
  pm.absorb = 1.0;
  double lw = interp_linear(rest_wavelengths, log_omega, 1, j, rest);
  double lya_z = (w - lya_wavelength) / lya_wavelength;                           // :117-119
  if (!meanflux) {
    double scaling = 1.0 - exp(-tau_0 * pow(1.0 + lya_z, beta)) + c_0;           // :144
    pm.om2 = exp(2.0 * lw) * (scaling * scaling);                                 // :142,146
  } else {
    // multi_dlas/process_qsos_multiple_dlas_meanflux.m:245-293
    double depth = tau_0 * pow(1.0 + lya_z, beta);                                // :245
    for (int l = 1; l < c_forest.num_forest_lines; ++l) {                         // :247-259
      double lyman_1pz = c_forest.wavelength[0] * (1.0 + lya_z) / c_forest.wavelength[l];
      if (lyman_1pz <= 1.0 + z_qso) depth = depth + (tau_0 * c_forest.tau_ratio[l]) * pow(lyman_1pz, beta);
    }
    double scaling = 1.0 - exp(-depth) + c_0;                                     // :261
    double om2 = exp(2.0 * lw) * (scaling * scaling);                             // :263
    double total = 0.0;
    for (int l = 0; l < c_forest.num_forest_lines; ++l) {                         // :269-283
      double zl = (w - c_forest.wavelength[l]) / c_forest.wavelength[l];          // :183-187
      if (l == 0 || !(zl > z_qso)) total = total + c_forest.kim_tau[l] * pow(1.0 + zl, c_forest.prev_beta);
    }
    pm.absorb = exp(-total);                                                      // :285
    pm.om2 = om2 * (pm.absorb * pm.absorb);                                       // :293
  }
  return pm;
}

// Entry p of the padded wavelength grid of process_qsos.m:168-176 for a window of n_u pixels starting at `wl_first`
// whose smallest / largest wavelengths have log10 lo / hi; entries past the reference's trailing pad continue the log
// grid.
__device__ __forceinline__ double padded_wavelength(int p, int n_u, const double* wl_first, double lo, double hi,
                                                    double pixel_spacing) {
  const int W3 = 3;
  if (p < W3) {
    // logspace(lo - 3 ps, lo - ps, 3) = 10.^linspace(a, b, 3)
    double a0 = lo - W3 * pixel_spacing, b0 = lo - pixel_spacing;
    double ex = (p == W3 - 1) ? b0 : a0 + p * ((b0 - a0) / (W3 - 1));
    return exp10(ex);
  }
  if (p < W3 + n_u) return wl_first[p - W3];
  int t = p - (W3 + n_u);   // 0,1,2 are the reference's trailing pad; beyond that: filler
  double a0 = hi + pixel_spacing, b0 = hi + W3 * pixel_spacing;
  double ex = (t == W3 - 1) ? b0 : a0 + t * ((b0 - a0) / (W3 - 1));
  return exp10(ex);
}

__global__ void __launch_bounds__(NTHREADS) prepare_quasars_kernel(PrepArgs a) {
  const int q = blockIdx.x, tid = threadIdx.x;
  const int64_t L = min(max((int64_t)a.lengths[q], (int64_t)0), a.L_max);   // a length beyond the padded row is clamped
  const double z_qso = a.z_qsos[q];
  const double* wl = a.wavelengths + q * a.L_max;
  const double* fl = a.flux + q * a.L_max;
  const double* nv = a.noise_variance + q * a.L_max;
  const uint8_t* pm = a.pixel_mask + q * a.L_max;

  __shared__ int s_first, s_last, s_n, s_nq, s_nd;
  __shared__ double s_minw, s_maxw, s_minu, s_maxu;
  __shared__ double red_min[NTHREADS / 32], red_max[NTHREADS / 32];
  if (tid == 0) { s_first = 1 << 30; s_last = -1; s_n = 0; s_nq = 0; s_nd = 0; }
  __syncthreads();

  // window / mask (process_qsos.m:102-110); min/max of used and of window wavelengths
  int first = 1 << 30, last = -1, n = 0;
  double minw = INFINITY, maxw = -INFINITY, minu = INFINITY, maxu = -INFINITY;
  for (int64_t i = tid; i < L; i += NTHREADS) {
    double w = wl[i];
    double rest = w / (1.0 + z_qso);
    bool inwin = (rest >= a.min_lambda) && (rest <= a.max_lambda);
    if (inwin) {
      first = min(first, (int)i); last = max(last, (int)i);
      minu = fmin(minu, w); maxu = fmax(maxu, w);
      if (!pm[i]) { n++; minw = fmin(minw, w); maxw = fmax(maxw, w); }
    }
  }
  // DLA existence prior counts (process_qsos.m:122-125)
  int nq = 0, nd = 0;
  const double zlim = z_qso + a.prior_z_qso_increase;
  for (int64_t i = tid; i < a.n_prior; i += NTHREADS) {
    bool less = a.prior_z_qsos[i] < zlim;
    nq += less; nd += (less && a.prior_dla_ind[i]);
  }
  atomicMin(&s_first, first); atomicMax(&s_last, last);
  atomicAdd(&s_n, n); atomicAdd(&s_nq, nq); atomicAdd(&s_nd, nd);
  auto block_minmax = [&](double vmin, double vmax, double& omin, double& omax) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      vmin = fmin(vmin, __shfl_xor_sync(0xffffffffu, vmin, o));
      vmax = fmax(vmax, __shfl_xor_sync(0xffffffffu, vmax, o));
    }
    __syncthreads();
    if ((tid & 31) == 0) { red_min[tid >> 5] = vmin; red_max[tid >> 5] = vmax; }
    __syncthreads();
    if (tid == 0) {
      for (int w = 1; w < NTHREADS / 32; ++w) { vmin = fmin(vmin, red_min[w]); vmax = fmax(vmax, red_max[w]); }
      omin = vmin; omax = vmax;
    }
  };
  block_minmax(minw, maxw, s_minw, s_maxw);
  block_minmax(minu, maxu, s_minu, s_maxu);
  __syncthreads();

  const int n_u = s_last >= s_first ? s_last - s_first + 1 : 0;
  const int n_used = s_n;
  const int NPIX = a.NPIX;
  double* lam = a.lam_pad + (int64_t)q * (NPIX + 8);
  double* lamh = a.lamh + (int64_t)q * (NPIX + 8);
  double* pix = a.pix + (int64_t)q * NPIX * 4;
  double* Mq = a.Mq + (int64_t)q * NPIX * a.k;
  // first padded wavelength (same expression as p = 0 below)
  const double lam_ref = n_used > 0 ? exp10(log10(s_minu) - 3 * a.pixel_spacing) : 1.0;

  if (tid == 0) {
    QuasarMeta m;
    m.lam_ref = lam_ref;
    m.n_u = n_u; m.n = n_used; m.nchunks = (n_u + KC - 1) / KC; m.first = s_first;
    // set_parameters.m:65-73
    m.max_z_dla = (s_maxw / a.lya_wavelength - 1.0) - a.max_z_cut;
    m.min_z_dla = fmax(s_minw / a.lya_wavelength - 1.0,
                       a.lyman_limit * (1.0 + z_qso) / a.lya_wavelength - 1.0 + a.min_z_cut);
    // process_qsos.m:128-131
    m.log_prior_dla = log((double)s_nd) - log((double)s_nq);
    m.prior_num_quasars = s_nq; m.prior_num_dlas = s_nd;
    m.log_prior_no_dla = log((double)(s_nq - s_nd)) - log((double)s_nq);
    if (n_used == 0) { m.nchunks = 0; m.min_z_dla = NAN; m.max_z_dla = NAN; }
    a.meta[q] = m;
  }
  if (n_used == 0) return;

  // padded wavelength grid (process_qsos.m:168-176); pixels past the end continue the log grid
  const double lo = log10(s_minu), hi = log10(s_maxu);
  for (int p = tid; p < NPIX + 8; p += NTHREADS) {
    const double v = padded_wavelength(p, n_u, wl + s_first, lo, hi, a.pixel_spacing);
    lam[p] = v;
    lamh[p] = log1p((v - lam_ref) / lam_ref) * a.inv_h;
  }

  // per-pixel model interpolation (process_qsos.m:138-146)
  for (int i = tid; i < NPIX; i += NTHREADS) {
    double y = 0.0, v = 1.0, mu = 0.0, om2 = 0.0, absorb = 1.0;
    bool used = false;
    int j = 0;
    double rest = 0.0;
    if (i < n_u) {
      int src = s_first + i;
      double w = wl[src];
      rest = w / (1.0 + z_qso);
      used = !pm[src] && (rest >= a.min_lambda) && (rest <= a.max_lambda);
      if (used) {
        y = fl[src]; v = nv[src];
        const PixelModel m = null_model_pixel(a.rest_wavelengths, a.mu, a.log_omega, a.n_rest, a.c_0, a.tau_0, a.beta,
                                              a.lya_wavelength, a.meanflux, w, rest, z_qso);
        j = m.j; om2 = m.om2; absorb = m.absorb;
        mu = m.mu * absorb;                                                          // :287 (exact when absorb = 1)
      }
    }
    pix[i * 4 + 0] = y; pix[i * 4 + 1] = v; pix[i * 4 + 2] = mu; pix[i * 4 + 3] = om2;
    for (int c = 0; c < a.k; ++c)
      Mq[(int64_t)i * a.k + c] = used ? interp_linear(a.rest_wavelengths, a.M + c, a.k, j, rest) * absorb : 0.0;   // :288
  }
}

// K0b: Gram operand P, chunked [Q][chunk][KC][BSTR]: columns pair_index(p,q) = M_ip M_iq, then the k
// columns of M itself (projection), zero padding elsewhere.
template <int K, int NSPLIT>
__global__ void __launch_bounds__(NTHREADS) build_gram_operand_kernel(const double* __restrict__ Mq,
                                                                      const QuasarMeta* __restrict__ meta,
                                                                      double* __restrict__ P, int NPIX,
                                                                      const int32_t* __restrict__ only_list, int q_offset) {
  using G = GramShape<K>;
  using SS = SplitShape<K, NSPLIT>;
  const int chunk = blockIdx.x;
  const int split = blockIdx.z;
  __shared__ double sM[KC][K + 1];
  // grid.y quasars of the batch from q_offset on, or the listed ones (grid.y slots stride over the list)
  const int nlist = only_list ? only_list[0] : (int)gridDim.y;
  for (int qi = blockIdx.y; qi < nlist; qi += gridDim.y) {
  const int q = only_list ? only_list[1 + qi] : qi + q_offset;
  if (chunk >= meta[q].nchunks) continue;
  __syncthreads();
  const double* src = Mq + ((int64_t)q * NPIX + (int64_t)chunk * KC) * K;
  for (int t = threadIdx.x; t < KC * K; t += NTHREADS) sM[t / K][t % K] = src[t];
  __syncthreads();
  // layout [q][split][chunk][KC][BSTR]
  double* dst = P + (((int64_t)q * NSPLIT + split) * (NPIX / KC) + chunk) * SS::CHUNK_DOUBLES;
  for (int t = threadIdx.x; t < SS::CHUNK_DOUBLES; t += NTHREADS) {
    int r = t / SS::BSTR, pos = t % SS::BSTR;
    // storage position -> local column: the two n8 tiles of a pair are interleaved so that one 16-byte
    // shared-memory load fetches a lane's B fragments of both (position 16 j + 2 g + t  <->  tile 2j + t, column g)
    int cl = pos;
    if (pos < SS::NCOLL) {
      const int j = pos / 16, w = pos % 16;
      if (2 * j + 1 < SS::NTL) cl = (2 * j + (w & 1)) * 8 + (w >> 1);
      else cl = (w < 8) ? 2 * j * 8 + w : SS::NCOLL;   // odd last tile: plain layout, rest padding
    }
    int c = split * SS::NCOLL + cl;          // global column
    double v = 0.0;
    if (cl < SS::NCOLL) {
      if (c < G::NPAIR) {
        // invert pair_index: find p with pair_index(p,p) <= c
        int p = 0;
        while (p + 1 < K && G::pair_index(p + 1, p + 1) <= c) ++p;
        int qq = p + (c - G::pair_index(p, p));
        v = sM[r][p] * sM[r][qq];
      } else if (c >= G::WT * 8 && c < G::WT * 8 + K) {
        v = sM[r][c - G::WT * 8];
      }
    }
    dst[t] = v;
  }
  }
}

// ------------------------------------------------------------------------------------------
// K1 (stand-alone): batched absorption profiles  A[s, i] = voigt(lambdas, z_s, N_s, num_lines)[i]
// grid = (S, ceil(n_out / 256))
__global__ void __launch_bounds__(NTHREADS) voigt_batch_kernel(const double* __restrict__ lambdas, int64_t num_points,
                                                               const double* __restrict__ zs,
                                                               const double* __restrict__ Ns, int num_lines,
                                                               double* __restrict__ profile) {
  __shared__ double s_raw[NTHREADS + 6];
  __shared__ double s_mult[MAX_LINES];
  const int64_t n_out = num_points - 6;
  const int64_t s = blockIdx.x;
  const int64_t i0 = (int64_t)blockIdx.y * NTHREADS;
  const double z = zs[s], N = Ns[s];
  if (threadIdx.x < num_lines) s_mult[threadIdx.x] = line_multiplier(threadIdx.x, z);
  __syncthreads();
  for (int t = threadIdx.x; t < NTHREADS + 6; t += NTHREADS) {
    int64_t p = i0 + t;
    if (p < num_points) {
      double tau = tau_sum_generic(lambdas[p], s_mult, 1, num_lines);
      s_raw[t] = exp_nonpos(-N * tau);                // voigt.c:291
    }
  }
  __syncthreads();
  int64_t i = i0 + threadIdx.x;
  if (i < n_out) {
    double acc = 0.0;
#pragma unroll
    for (int t = 0; t < 7; ++t) acc = fma(s_raw[threadIdx.x + t], c_lines.ip[t], acc);   // voigt.c:297-299
    profile[s * n_out + i] = acc;
  }
}

// ------------------------------------------------------------------------------------------
// K1+K2+K3 fused: per-(quasar, sample-tile) log-likelihoods.
struct LoglikArgs {
  const QuasarMeta* meta;
  const double* lam_pad;      // [Q x (NPIX + 8)]
  const double* lamh;         // [Q x (NPIX + 8)]  grid positions for the rest-frame table
  RestTable rt;               // rest-frame table of tau / N (coef == nullptr: direct evaluation everywhere)
  const int32_t* order;       // [S] samples in ascending redshift offset (tile position -> sample); nullptr = identity
  const double* pix;          // [Q x NPIX x 4]
  const double* P;            // [Q x NPIX/KC x KC x BSTR]
  const double* offset_samples;
  const double* nhi_samples;
  int64_t S;                  // number of DLA samples; sample index S is the null model (absorption == 1)
  int num_lines;
  int NPIX;
  double* sample_log_likelihoods;   // [Q x S] (row stride sll_stride)
  double* log_likelihoods_no_dla;   // [Q]; nullptr: no null-model slot (tiles cover S samples only)
  int64_t sll_stride;               // elements between consecutive quasars' rows of sample_log_likelihoods
  // multi-DLA levels (...meanflux.m:337-381): the convolved absorption of every sample is cached at level 1
  // (MODE 1) and levels >= 2 (MODE 2) multiply cached rows instead of re-evaluating Voigt profiles
  double* acache;                   // [Q x S x NPIX]
  const int32_t* partners;          // [Q x 3 x S] 0-based base_sample_inds; level l uses rows 0..l-2
  int num_partners;
  const int32_t* active;            // [Q] or nullptr; 0 = quasar finished early (:460-464) -> NaN
  int q_offset;                     // dla_loglik_ws_kernel: first quasar of the batch this launch covers (grid.y counts from it)
  const int32_t* only_list;         // dla_loglik_ws_list_kernel: {count, q_0, q_1, ...}, the quasars to process -- the INT8
                                    // path's FP64 fallback for zero-noise-variance pixels
  // column-split ranks (NSPLIT > 1): accumulators and per-sample scalars leave through global memory
  double* gram;                     // [Q x rows x NCOL], rows = sample tiles * 64
  double* qld;                      // [Q x rows x 2]  (sum r^2/d, sum log d)
  int64_t gram_rows;
};


// Tile position -> sample index (samples are processed in ascending redshift so that the warps of a CTA look up
// neighbouring cells of the rest-frame table; results go back to the caller's order).
__device__ __forceinline__ int64_t sample_at(const LoglikArgs& args, int64_t pos) {
  return args.order ? (int64_t)args.order[pos] : pos;
}

// One k4-step of the contraction for one warp: NT n8 tiles, B fragments fetched pairwise with 16-byte loads
// from the pair-interleaved P chunk row `brow2` (= chunk + k * BSTR + 2 * gid).
template <int NT, int WT>
__device__ __forceinline__ void dmma_k4_step(double (&acc)[NT][2], double aw, double au, const double* brow2, int tile0,
                                             int gid) {
#pragma unroll
  for (int j = 0; j < NT / 2; ++j) {
    const double2 b = *reinterpret_cast<const double2*>(brow2 + j * 16);
    dmma_884(acc[2 * j][0], acc[2 * j][1], (tile0 + 2 * j) < WT ? aw : au, b.x);
    dmma_884(acc[2 * j + 1][0], acc[2 * j + 1][1], (tile0 + 2 * j + 1) < WT ? aw : au, b.y);
  }
  if (NT % 2) {
    const double b = brow2[(NT / 2) * 16 - gid];   // plain layout of the odd last tile: position 16 (NT/2) + gid
    dmma_884(acc[NT - 1][0], acc[NT - 1][1], (tile0 + NT - 1) < WT ? aw : au, b);
  }
}

template <int K, int CSTR>
__device__ __forceinline__ void factor_staged(double* Cs, const double* s_q, const double* s_ld, int row0, int lane,
                                              const QuasarMeta& meta, const LoglikArgs& args, int q, int64_t s0);

// Epilogue shared by the fused kernels: stage one warp's 8 x NCOL accumulator tile through shared memory as
// an augmented upper triangle and factorise it (K3).  `row0` = first sample row of this warp inside the CTA.
template <int K, int NT, int CSTR>
__device__ __forceinline__ void stage_and_factor(double (&acc)[NT][2], double* Cs, const double* s_q, const double* s_ld,
                                                 int row0, int lane, const QuasarMeta& meta, const LoglikArgs& args,
                                                 int q, int64_t s0) {
  const int gid = lane >> 2, tig = lane & 3;
  const int64_t S = args.S;
  // C fragment: lane holds row gid, columns 2 tig, 2 tig + 1 of each n8 tile
#pragma unroll
  for (int ni = 0; ni < NT; ++ni) {
    const int i0 = stage_index_table<K>()[ni * 8 + tig * 2], i1 = stage_index_table<K>()[ni * 8 + tig * 2 + 1];
    if (i0 >= 0) Cs[i0 * CSTR + row0 + gid] = acc[ni][0];
    if (i1 >= 0) Cs[i1 * CSTR + row0 + gid] = acc[ni][1];
  }
  __syncwarp();
  factor_staged<K, CSTR>(Cs, s_q, s_ld, row0, lane, meta, args, q, s0);
}

// K3: Cholesky of B = I + C (upper, R'R = B) from the staged augmented triangle, with the projected vector
// g as column K (forward substitution for free), log-det, quadratic form.  One warp factorises the 8 samples
// row0..row0+7: four lanes per sample; for row p the columns q = p+1 .. K are dealt round-robin to the quad.
// Fully unrolled: every index is an immediate.
template <int K, int CSTR>
__device__ __forceinline__ void factor_staged(double* Cs, const double* s_q, const double* s_ld, int row0, int lane,
                                              const QuasarMeta& meta, const LoglikArgs& args, int q, int64_t s0) {
  const int64_t S = args.S;
  {
    const int sl = row0 + (lane >> 2);          // sample handled by this lane quad
    const int l4 = lane & 3;
    double* Bs = Cs + sl;                              // entry (p, q) at Bs[aug_index<K>(p, q) * CSTR]
    double prod0 = 1.0, prod1 = 1.0;
#pragma unroll
    for (int p = 0; p < K; ++p) {
      double colp[K];                                  // R(r, p), r < p
#pragma unroll
      for (int r = 0; r < p; ++r) colp[r] = Bs[aug_index<K>(r, p) * CSTR];
      double dpp = Bs[aug_index<K>(p, p) * CSTR] + 1.0;                       // log_mvnpdf_low_rank.m:23
#pragma unroll
      for (int r = 0; r < p; ++r) dpp = fma(-colp[r], colp[r], dpp);
      if (p < K / 2) prod0 *= dpp; else prod1 *= dpp;                       // log det B = log prod R(p,p)^2   :30
      const double inv = rsqrt(dpp);
#pragma unroll
      for (int j = 0; j < (K - p + 3) / 4; ++j) {
        const int qq = p + 1 + l4 + 4 * j;
        if (qq <= K) {
          double* dst = Bs + (aug_index<K>(p, p) + (qq - p)) * CSTR;
          double v = *dst;
#pragma unroll
          for (int r = 0; r < p; ++r) v = fma(-colp[r], Bs[(aug_index<K>(r, r) + (qq - r)) * CSTR], v);
          *dst = v * inv;
        }
      }
      __syncwarp();
    }
    double zsum = 0.0;                                 // |R'^-1 g|^2: column K now holds z
#pragma unroll
    for (int p = 0; p < K; ++p) { const double zp = Bs[aug_index<K>(p, K) * CSTR]; zsum = fma(zp, zp, zsum); }
    if (l4 == 0) {
      const double quad = s_q[sl] - zsum;                                   // y' K^-1 y                 :28
      const double logdet = s_ld[sl] + log(prod0) + log(prod1);             //                           :30
      const double lp = -0.5 * (quad + logdet + (double)meta.n * LOG_2PI);  //                           :32
      const int64_t s = s0 + sl;
      if (s < S) args.sample_log_likelihoods[(int64_t)q * args.sll_stride + sample_at(args, s)] = lp;
      else if (s == S && args.log_likelihoods_no_dla) args.log_likelihoods_no_dla[q] = lp;
    }
  }
}

// MODE 0: single-DLA / sub-DLA pass;  MODE 1: same, and the convolved absorption rows are stored in
// args.acache;  MODE 2: multi-DLA level >= 2, absorption = product of cached rows (sample and partners).
// ------------------------------------------------------------------------------------------
// Warp-specialised schedule.
//
// Measured on B200 (profiles/r01_fp64_mix.txt, r01_dmma_loop.txt): DMMA and DFMA share one pipe per SM
// sub-partition and its arbiter favours DMMA -- while two warps of a sub-partition issue DMMA, DFMA warps
// there do not progress at all; with one DMMA warp they get 31 % and the DMMA stream 62 %.  A lone DMMA warp
// that also fetches its fragments from shared memory reaches only 78 % of the pipe, two warps reach ~100 %.
// Tried and measured (ms per 296 quasars): 1 consumer + 2 producers per sub-partition 89.6-91.2 (shipped);
// 2 consumers + 1 producer 132.5 (the producer only runs while both consumers wait, and a lone warp's
// profile arithmetic is latency-bound); 2 consumers + 2 producers with setmaxnreg 97.7.  Roles, per CTA of
// WS_CONSUMERS x 8 samples of one quasar (defaults: 4 consumers, 8 producers, 32 samples, 168 registers):
//   * CONSUMER warps (0..NC-1, one per sub-partition): consumer c runs the FP64 DMMA contraction of sample
//     rows 8c..8c+7 (one m8 tile x all n8 tiles, accumulators in 120 registers) against the shared P chunk;
//   * PRODUCER warps (NC.., two per sub-partition): each makes 4 of a consumer's 8 rows per chunk -- Voigt raw
//     profile, instrument convolution, weights w = a^2/d, u = a (y - a mu)/d, lane = pixel -- and accumulates
//     the per-sample scalars sum r^2/d and prod d.
// Rows travel through 2-stage full/empty mbarriers per consumer; P chunks arrive by 1-D TMA bulk copies into
// a double buffer re-armed by the last consumer to finish.  No CTA-wide barrier in the main loop.
constexpr int RAWS = KC + 8;      // raw-profile row: 6 carried-over pixels + KC new ones (+2 pad)
#ifndef GPDLA_WS_CONSUMERS
#define GPDLA_WS_CONSUMERS 4
#define GPDLA_WS_PRODUCERS 8
#endif
constexpr int WS_CONSUMERS = GPDLA_WS_CONSUMERS, WS_PRODUCERS = GPDLA_WS_PRODUCERS;
constexpr int WS_THREADS = 32 * (WS_CONSUMERS + WS_PRODUCERS);   // 384 -> 168 registers per thread
#ifndef GPDLA_WS_STAGES
#define GPDLA_WS_STAGES 2
#endif
constexpr int WS_STAGES = GPDLA_WS_STAGES;   // operand-row stages between producer and consumer

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// tau / N of SPB samples at one wavelength by direct evaluation of the line sum (lane = pixel)   voigt.c:282-290:
// branch-free wing formula for all samples, then the exact routine for the lanes within X0 Doppler widths of a core.
//   mymult[j * mstride + ss]: line multipliers (voigt.c:279)
template <int SPB>
struct TauRow { double t[SPB]; };

// Kept out of line on purpose: the direct evaluation runs in < 10 % of the chunks but needs far more registers than
// the rest of the producer loop; inlined, it costs the common path its instruction-level parallelism (measured: the
// whole kernel 20 % slower).
template <int NL, int SPB>
__device__ __noinline__ TauRow<SPB> tau_direct(double lambda, const double* mymult, int mstride, int num_lines) {
  TauRow<SPB> out;
  double (&tau)[SPB] = out.t;
  if (NL == 3) {
    const int lane = threadIdx.x & 31;
    unsigned cm[SPB], any = 0;
#pragma unroll
    for (int ss = 0; ss < SPB; ++ss) {
      bool core;
      tau[ss] = tau_sum_3_wing(lambda, mymult[ss], mymult[mstride + ss], mymult[2 * mstride + ss], core);
      cm[ss] = __ballot_sync(0xffffffffu, core);
      any |= cm[ss];
    }
    if (any) {   // warp-uniform
      // The (sample, pixel) pairs within X0 Doppler widths of a line core -- at most 7 pixels per sample, and the SPB
      // samples of a warp are neighbours in redshift, so they all arrive in this chunk -- are dealt out one per lane
      // and evaluated by ONE pass of the exact routine instead of SPB divergent passes with 7 active lanes each.
      int off[SPB + 1];
      off[0] = 0;
#pragma unroll
      for (int ss = 0; ss < SPB; ++ss) off[ss + 1] = off[ss] + __popc(cm[ss]);
      if (off[SPB] <= 32) {
        int ss_i = 0;
#pragma unroll
        for (int ss = 1; ss < SPB; ++ss) ss_i = (lane >= off[ss]) ? ss : ss_i;
        unsigned mask_i = cm[0];
        int off_i = 0;
#pragma unroll
        for (int ss = 1; ss < SPB; ++ss) { mask_i = (ss_i == ss) ? cm[ss] : mask_i; off_i = (ss_i == ss) ? off[ss] : off_i; }
        const bool have = lane < off[SPB];
        const int src = have ? (int)__fns(mask_i, 0, lane - off_i + 1) : 0;       // pixel lane of this lane's pair
        const double lam_i = __shfl_sync(0xffffffffu, lambda, src);
        const double t = tau_sum_3_exact(lam_i, mymult[ss_i], mymult[mstride + ss_i], mymult[2 * mstride + ss_i]);
        const unsigned below = (1u << lane) - 1u;
#pragma unroll
        for (int ss = 0; ss < SPB; ++ss) {
          const double v = __shfl_sync(0xffffffffu, t, (off[ss] + __popc(cm[ss] & below)) & 31);
          if ((cm[ss] >> lane) & 1u) tau[ss] = v;
        }
      } else {
#pragma unroll
        for (int ss = 0; ss < SPB; ++ss)
          if ((cm[ss] >> lane) & 1u)
            tau[ss] = tau_sum_3_exact(lambda, mymult[ss], mymult[mstride + ss], mymult[2 * mstride + ss]);
      }
    }
  } else {
#pragma unroll
    for (int ss = 0; ss < SPB; ++ss) tau[ss] = tau_sum_generic(lambda, mymult + ss, mstride, num_lines);
  }
  return out;
}

// tau / N of SPB samples from the cell fetched for this lane; returns true (warp-uniform) when some lane's cell is
// one of those left to direct evaluation.  All 32 lanes must call this together.
template <int SPB>
__device__ __forceinline__ bool tau_from_cell(const RestCell& rc, const double* myK, double (&tau)[SPB]) {
  unsigned worst = 0;
#pragma unroll
  for (int ss = 0; ss < SPB; ++ss) {
    tau[ss] = rest_table_eval(rc, myK[ss]);
    worst = max(worst, (unsigned)__double2hiint(tau[ss]));
  }
  return __any_sync(0xffffffffu, worst >= 0x7ff00000u);
}

// tau / N of SPB samples, each from its own cell (samples too far apart in redshift to share one).  Out of line like the
// direct evaluation: a mode for sparse sample sets that must not cost the common path registers.
template <int SPB>
__device__ __noinline__ TauRow<SPB> tau_own_cells(const RestTable& rt, double lh, const double* myK) {
  TauRow<SPB> out;
#pragma unroll
  for (int ss = 0; ss < SPB; ++ss) {
    RestCell rc;
    const double K = myK[ss];
    rest_table_fetch(rt, lh, K, rc);
    out.t[ss] = rest_table_eval(rc, K);
  }
  return out;
}

// tau / N of the SPB samples of a group at one wavelength.  `tab_mode` (see group_cell): 1 = the group's common cell of
// the rest-frame table, 2 = the samples are too far apart in redshift to share a cell (few samples per quasar): one cell
// per sample, 0 = no table.  Where a cell is near a line centre the whole warp evaluates directly.  The coefficient
// loads hit L1 when the warps of a CTA work on neighbouring redshifts (a line holds 16 cells and is used by every warp
// for one or two chunks); all 32 lanes must call this together.
// `cell`: the group's cell when the caller fetched it ahead of time (tab_mode 1 only), else nullptr
template <int NL, int SPB>
__device__ __forceinline__ void tau_samples(const RestTable& rt, int tab_mode, double K_mid, double lambda, double lh,
                                            const double* mymult, int mstride, const double* myK, int num_lines,
                                            double (&tau)[SPB], const RestCell* cell = nullptr) {
  bool direct = tab_mode == 0;
  if (tab_mode == 1) {
    RestCell rc;
    if (cell) rc = *cell;
    else rest_table_fetch(rt, lh, K_mid, rc);
    direct = tau_from_cell<SPB>(rc, myK, tau);
  } else if (tab_mode == 2) {
    const TauRow<SPB> r = tau_own_cells<SPB>(rt, lh, myK);
    unsigned worst = 0;
#pragma unroll
    for (int ss = 0; ss < SPB; ++ss) { tau[ss] = r.t[ss]; worst = max(worst, (unsigned)__double2hiint(tau[ss])); }
    direct = __any_sync(0xffffffffu, worst >= 0x7ff00000u);
  }
  if (direct) {
    const TauRow<SPB> r = tau_direct<NL, SPB>(lambda, mymult, mstride, num_lines);
#pragma unroll
    for (int ss = 0; ss < SPB; ++ss) tau[ss] = r.t[ss];
  }
}

// raw absorption exp(-N tau)   voigt.c:291.  All shared-memory loads come before the caller's first store: the
// compiler cannot prove that the per-sample arrays and the raw rows do not alias, and a load stuck behind a store
// would serialise the SPB exponentials.
template <int SPB, bool EXP_TABLE = (GPDLA_EXP_TABLE != 0)>
__device__ __forceinline__ void raw_from_tau(const double (&tau)[SPB], const double* mynhi, double (&e)[SPB]) {
#pragma unroll
  for (int ss = 0; ss < SPB; ++ss) e[ss] = -mynhi[ss] * tau[ss];
#pragma unroll
  for (int ss = 0; ss < SPB; ++ss) e[ss] = exp_nonpos<EXP_TABLE>(e[ss]);
}

// K_mid of a group of SPB consecutive tile rows (their table offsets in myK) and how the table serves them: 1 = one
// cell for the group, 2 = one cell per sample, 0 = table disabled
template <int SPB>
__device__ __forceinline__ int group_cell(const RestTable& rt, const double* myK, double& K_mid) {
  double lo = myK[0], hi = myK[0];
#pragma unroll
  for (int ss = 1; ss < SPB; ++ss) { lo = fmin(lo, myK[ss]); hi = fmax(hi, myK[ss]); }
  K_mid = 0.5 * (lo + hi);
  return rt.coef == nullptr ? 0 : ((hi - lo) <= RT_MAX_SPREAD ? 1 : 2);
}

template <int K, int NSPLIT>
struct WsConfig {
  using G = GramShape<K>;
  using SS = SplitShape<K, NSPLIT>;
  static constexpr int SPW = 8;                         // samples per consumer = one m8 tile
  static constexpr int SPB = 4;                         // samples per producer batch
  static constexpr int TS = WS_CONSUMERS * SPW;         // 64 samples per CTA
  static constexpr int SPP = TS / WS_PRODUCERS;         // 16 samples per producer
  static constexpr size_t B_BYTES = 2ull * SS::CHUNK_DOUBLES * 8;
  static constexpr size_t A_BYTES = (size_t)WS_STAGES * 2 * TS * ASTR * 8;     // W and U, WS_STAGES stages
  static constexpr size_t RAW_BYTES = (size_t)TS * RAWS * 8;
  static constexpr int CSTR = TS + 4;
  static constexpr size_t C_BYTES = (size_t)((K + 1) * (K + 2) / 2) * CSTR * 8;
  static_assert(NSPLIT > 1 || C_BYTES <= B_BYTES + A_BYTES, "epilogue staging must fit");
  static_assert(SS::NTL * 4 + 40 <= 168, "accumulators must fit in the consumer's registers");
  static constexpr int NBAR = 2 + 2 * WS_STAGES * WS_CONSUMERS;
  __host__ __device__ static constexpr size_t smem_bytes(int num_lines) {
    return B_BYTES + A_BYTES + RAW_BYTES + (size_t)TS * (num_lines + 4) * 8 + NBAR * 8 + 64 + 4 * TS * 4;
  }
};

__device__ __forceinline__ void mbar_inval(uint64_t* bar) {
  asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// One (quasar, sample tile, column split) of the warp-specialised FP64 kernel.
template <int K, int NL, int MODE, int NSPLIT>
__device__ __forceinline__ void ws_tile(const LoglikArgs& args, const int q) {
  using Cfg = WsConfig<K, NSPLIT>;
  using G = GramShape<K>;
  using SS = SplitShape<K, NSPLIT>;
  constexpr int TS = Cfg::TS, SPW = Cfg::SPW, SPB = Cfg::SPB, SPP = Cfg::SPP, NT = SS::NTL, CSTR = Cfg::CSTR;
  const int split = (NSPLIT > 1) ? blockIdx.z : 0;
  const int tile0 = split * SS::NTL;
  const QuasarMeta meta = args.meta[q];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int64_t s0 = (int64_t)blockIdx.x * TS;
  const int64_t S = args.S;

  // nothing usable in this spectrum (process_qsos.m:74-82), or the level loop already ended for this quasar
  // (...meanflux.m:460-464): NaN results
  if (meta.nchunks == 0 || (args.active != nullptr && args.active[q] == 0)) {
    for (int i = tid; i < TS && split == 0; i += WS_THREADS) {
      int64_t s = s0 + i;
      if (s < S) args.sample_log_likelihoods[(int64_t)q * args.sll_stride + s] = NAN;
      else if (s == S && args.log_likelihoods_no_dla) args.log_likelihoods_no_dla[q] = NAN;
    }
    return;
  }

  extern __shared__ __align__(128) unsigned char smem_raw[];
  double* Bt = reinterpret_cast<double*>(smem_raw);                       // [2][KC][BSTR]
  double* Wt = reinterpret_cast<double*>(smem_raw + Cfg::B_BYTES);        // [WS_STAGES][TS][ASTR]
  double* Ut = Wt + WS_STAGES * TS * ASTR;                                // [WS_STAGES][TS][ASTR]
  double* rawbuf = Ut + WS_STAGES * TS * ASTR;                            // [TS][RAWS]
  double* s_nhi = rawbuf + TS * RAWS;                                     // [TS]
  double* s_q = s_nhi + TS;                                               // [TS]   sum r^2/d
  double* s_ld = s_q + TS;                                                // [TS]   sum log d
  double* s_mult = s_ld + TS;                                             // [num_lines][TS]
  const int num_lines = (NL > 0) ? NL : args.num_lines;
  double* s_K = s_mult + (size_t)TS * num_lines;                           // [TS]   rest-frame table offsets
  uint64_t* bar_p = reinterpret_cast<uint64_t*>(s_K + TS);                 // P chunk full[2]
  uint64_t* bar_full = bar_p + 2;                                          // [consumer][stage] rows ready
  uint64_t* bar_empty = bar_full + WS_STAGES * WS_CONSUMERS;               // [consumer][stage] rows consumed
  int* s_done = reinterpret_cast<int*>(bar_empty + WS_STAGES * WS_CONSUMERS);   // [2] consumers done with P buffer
  int* s_part = s_done + 2;                                                // [3][TS] partner samples (MODE 2)
  int* s_so = s_part + 3 * TS;                                             // [TS]   sample index of every tile row
  double* Cs = reinterpret_cast<double*>(smem_raw);                       // epilogue: [entries][CSTR]

  for (int i = tid; i < TS; i += WS_THREADS) {                             // per-sample parameters
    const int64_t s = s0 + i;
    const bool is_null = s >= S;
    const int64_t so = sample_at(args, is_null ? S - 1 : s);   // the null-model slot borrows a redshift (a == 1 anyway)
    const double z = __dadd_rn(meta.min_z_dla, __dmul_rn(meta.max_z_dla - meta.min_z_dla, args.offset_samples[so]));
    s_nhi[i] = is_null ? -1.0 : args.nhi_samples[so];    // negative marks the null-model slot
    s_ld[i] = 0.0;
    s_K[i] = rest_table_offset(args.rt, z, meta.lam_ref);
    s_so[i] = (int)so;
    for (int j = 0; j < num_lines; ++j) s_mult[j * TS + i] = line_multiplier(j, z);
    if (MODE == 2) {
      for (int j = 0; j < args.num_partners; ++j)
        s_part[j * TS + i] = is_null ? 0 : args.partners[((int64_t)q * 3 + j) * S + so];
    }
  }
  const double* Pq = args.P + ((int64_t)q * NSPLIT + split) * (args.NPIX / KC) * SS::CHUNK_DOUBLES;
  constexpr uint32_t CHUNK_BYTES = SS::CHUNK_DOUBLES * 8;
  if (tid == 0) {
    mbar_init(&bar_p[0], 1);
    mbar_init(&bar_p[1], 1);
    for (int i = 0; i < WS_STAGES * WS_CONSUMERS; ++i) { mbar_init(&bar_full[i], 64); mbar_init(&bar_empty[i], 32); }
    s_done[0] = 0; s_done[1] = 0;
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    mbar_expect_tx(&bar_p[0], CHUNK_BYTES);
    tma_load_1d(Bt, Pq, CHUNK_BYTES, &bar_p[0]);
    if (meta.nchunks > 1) {
      mbar_expect_tx(&bar_p[1], CHUNK_BYTES);
      tma_load_1d(Bt + SS::CHUNK_DOUBLES, Pq + SS::CHUNK_DOUBLES, CHUNK_BYTES, &bar_p[1]);
    }
  }
  __syncthreads();

  double acc[NT][2];   // consumer accumulators (dead in producers)

  if (warp >= WS_CONSUMERS) {
    // =========================================================================== PRODUCER
    const int pr = warp - WS_CONSUMERS;
    const double* lam = args.lam_pad + (int64_t)q * (args.NPIX + 8);
    const double* pix = args.pix + (int64_t)q * args.NPIX * 4;
    double* const cache_q = (MODE != 0) ? args.acache + (int64_t)q * S * args.NPIX : nullptr;
    // the CTA's 2 * WS_CONSUMERS batches of 4 sample rows are dealt round-robin to the producers:
    // local batch b of producer pr is global batch j = pr + b * WS_PRODUCERS = rows 4 (j / NC) .. +4 of consumer j % NC
    auto batch_consumer = [&](int b) { return (pr + b * WS_PRODUCERS) % WS_CONSUMERS; };
    auto batch_row0 = [&](int b) { return batch_consumer(b) * SPW + ((pr + b * WS_PRODUCERS) / WS_CONSUMERS) * SPB; };

    // raw (unconvolved) absorption of 4 samples (rows row0..row0+3) at one wavelength    voigt.c:282-292
    const double* lamh = args.lamh + (int64_t)q * (args.NPIX + 8);
    auto eval_raw = [&](int row0, double lambda, double lh, double (&e)[SPB]) {
      double tau[SPB], K_mid;
      const int tab_mode = group_cell<SPB>(args.rt, s_K + row0, K_mid);
      tau_samples<NL, SPB>(args.rt, tab_mode, K_mid, lambda, lh, s_mult + row0, TS, s_K + row0, num_lines, tau);
      raw_from_tau<SPB>(tau, s_nhi + row0, e);
    };
    if (MODE != 2) {   // leading pad pixels p = 0..5
      const double lambda0 = lam[lane < 6 ? lane : 5], lh0 = lamh[lane < 6 ? lane : 5];
#pragma unroll
      for (int b = 0; b < SPP / SPB; ++b) {
        double e[SPB];
        eval_raw(batch_row0(b), lambda0, lh0, e);
        if (lane < 6) {
#pragma unroll
          for (int ss = 0; ss < SPB; ++ss) rawbuf[(batch_row0(b) + ss) * RAWS + lane] = e[ss];
        }
      }
    }
    double qacc[SPP], ldm[SPP];
    int lde[SPP];
#pragma unroll
    for (int ss = 0; ss < SPP; ++ss) { qacc[ss] = 0.0; ldm[ss] = 1.0; lde[ss] = 0; }

    // pixel data of the next chunk is fetched one chunk ahead (global/L2 latency off the critical path)
    double lambda_n = lam[6 + lane], lh_n = lamh[6 + lane];
    double2 p01n = *reinterpret_cast<const double2*>(pix + (int64_t)lane * 4);
    double2 p23n = *reinterpret_cast<const double2*>(pix + (int64_t)lane * 4 + 2);
    for (int c = 0; c < meta.nchunks; ++c) {
      const int stage = c % WS_STAGES;
      const int i = c * KC + lane;
      const double lambda = lambda_n, lh = lh_n;
      const double y = p01n.x, v = p01n.y, mu = p23n.x, om2 = p23n.y;
      if (c + 1 < meta.nchunks) {
        lambda_n = lam[i + KC + 6];
        lh_n = lamh[i + KC + 6];
        p01n = *reinterpret_cast<const double2*>(pix + (int64_t)(i + KC) * 4);
        p23n = *reinterpret_cast<const double2*>(pix + (int64_t)(i + KC) * 4 + 2);
      }
#pragma unroll
      for (int b = 0; b < SPP / SPB; ++b) {
        const int cons = batch_consumer(b), row0 = batch_row0(b);
        double* myraw = rawbuf + row0 * RAWS;
        double a[SPB];
        if (MODE != 2) {
          // ---- raw profile for the KC new padded pixels, then the instrument convolution (voigt.c:297-299)
          double e[SPB];
          eval_raw(row0, lambda, lh, e);
#pragma unroll
          for (int ss = 0; ss < SPB; ++ss) myraw[ss * RAWS + 6 + lane] = e[ss];
          __syncwarp();
          double carry[SPB];
#pragma unroll
          for (int ss = 0; ss < SPB; ++ss) {
            const double* rb = myraw + ss * RAWS;
            double acc_a = 0.0;
#pragma unroll
            for (int t = 0; t < 6; ++t) acc_a = fma(rb[lane + t], c_lines.ip[t], acc_a);
            acc_a = fma(e[ss], c_lines.ip[6], acc_a);   // the lane's own pixel is still in its register
            carry[ss] = rb[KC + (lane < 6 ? lane : 0)];
            a[ss] = (__double2hiint(s_nhi[row0 + ss]) < 0) ? 1.0 : acc_a;   // null model (N marked negative)
          }
          __syncwarp();
          if (lane < 6) {
#pragma unroll
            for (int ss = 0; ss < SPB; ++ss) myraw[ss * RAWS + lane] = carry[ss];   // last 6 pixels -> front of the row
          }
          if (MODE == 1 && split == 0) {   // keep the level-1 absorption rows for the higher multi-DLA levels
#pragma unroll
            for (int ss = 0; ss < SPB; ++ss)
              if (s0 + row0 + ss < S) cache_q[(int64_t)s_so[row0 + ss] * args.NPIX + i] = a[ss];
          }
        } else {
          // absorption = voigt(sample) .* voigt(partner 1) .* ...   (...meanflux.m:342-351), from the cache
#pragma unroll
          for (int ss = 0; ss < SPB; ++ss) a[ss] = cache_q[(int64_t)s_so[row0 + ss] * args.NPIX + i];
          for (int j = 0; j < args.num_partners; ++j) {
            double bb[SPB];
#pragma unroll
            for (int ss = 0; ss < SPB; ++ss) bb[ss] = cache_q[(int64_t)s_part[j * TS + row0 + ss] * args.NPIX + i];
#pragma unroll
            for (int ss = 0; ss < SPB; ++ss) a[ss] = a[ss] * bb[ss];
          }
        }
        // ---- weights into the consumer's operand rows of this stage, once it has released them
        mbar_wait(&bar_empty[cons * WS_STAGES + stage], ((c / WS_STAGES) & 1) ^ 1);
        double* dW = Wt + (stage * TS + row0) * ASTR + lane;
        double* dU = Ut + (stage * TS + row0) * ASTR + lane;
#pragma unroll
        for (int ss = 0; ss < SPB; ++ss) {
          const double a2 = a[ss] * a[ss];
          const double d = fma(a2, om2, v);                // dla_omega2 + noise variance  (process_qsos.m:194,198)
          const double rd = fast_rcp(d);
          const double r = fma(-a[ss], mu, y);             // y - dla_mu
          const double t1 = r * rd;
          dW[ss * ASTR] = a2 * rd;
          dU[ss * ASTR] = a[ss] * t1;
          qacc[b * SPB + ss] = fma(r, t1, qacc[b * SPB + ss]);
          ldm[b * SPB + ss] *= d;
        }
        mbar_arrive(&bar_full[cons * WS_STAGES + stage]);
      }
      if ((c & 7) == 7) {   // keep the running products of d in range: move their exponents to integers
#pragma unroll
        for (int ss = 0; ss < SPP; ++ss) {
          int hi = __double2hiint(ldm[ss]);
          int e2 = ((hi >> 20) & 0x7ff) - 1023;
          lde[ss] += e2;
          ldm[ss] = __hiloint2double(hi - (e2 << 20), __double2loint(ldm[ss]));
        }
      }
    }
#pragma unroll
    for (int b = 0; b < SPP / SPB; ++b)
#pragma unroll
      for (int ss = 0; ss < SPB; ++ss) {   // per-sample scalars: sum r^2/d and sum log d
        const double qs = warp_sum(qacc[b * SPB + ss]);
        const double ld = warp_sum(log(ldm[b * SPB + ss]) + (double)lde[b * SPB + ss] * 0.693147180559945309417);
        if (lane == 0) { s_q[batch_row0(b) + ss] = qs; s_ld[batch_row0(b) + ss] = ld; }
      }
  } else {
    // =========================================================================== CONSUMER
#pragma unroll
    for (int ni = 0; ni < NT; ++ni) acc[ni][0] = acc[ni][1] = 0.0;
    const int gid = lane >> 2, tig = lane & 3;
    const double* rW0 = Wt + (warp * SPW + gid) * ASTR + tig;
    const double* rU0 = Ut + (warp * SPW + gid) * ASTR + tig;
    for (int c = 0; c < meta.nchunks; ++c) {
      const int stage = c % WS_STAGES;           // operand-row stage
      const int pbuf = c & 1;                    // P chunk buffer
      mbar_wait(&bar_full[warp * WS_STAGES + stage], (c / WS_STAGES) & 1);
      mbar_wait(&bar_p[pbuf], (c >> 1) & 1);
      const double* Bc = Bt + pbuf * SS::CHUNK_DOUBLES + tig * SS::BSTR + 2 * gid;
      const double* rW = rW0 + stage * TS * ASTR;
      const double* rU = rU0 + stage * TS * ASTR;
      // FP64 tensor-core contraction  acc += [W|U] (8 x KC) . P_chunk (KC x NCOL)
#pragma unroll
      for (int ks = 0; ks < KC / 4; ++ks) {
        const double aw = rW[ks * 4];
        const double au = rU[ks * 4];
        dmma_k4_step<NT, G::WT>(acc, aw, au, Bc + ks * 4 * SS::BSTR, tile0, gid);
      }
      mbar_arrive(&bar_empty[warp * WS_STAGES + stage]);
      __syncwarp();
      // release the P buffer; the last consumer to finish this chunk re-arms it with chunk c + 2
      if (lane == 0 && c + 2 < meta.nchunks) {
        const int done = atomicAdd(&s_done[pbuf], 1);
        if (done == WS_CONSUMERS - 1) {
          s_done[pbuf] = 0;
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          mbar_expect_tx(&bar_p[pbuf], CHUNK_BYTES);
          tma_load_1d(Bt + pbuf * SS::CHUNK_DOUBLES, Pq + (int64_t)(c + 2) * SS::CHUNK_DOUBLES, CHUNK_BYTES,
                      &bar_p[pbuf]);
        }
      }
    }
  }
  __syncthreads();   // all operand/P buffers are dead -> the staging area may alias them; s_q, s_ld are final
  if (tid == 0) {    // the barriers are re-initialised if this CTA goes on to another quasar (only_list)
    mbar_inval(&bar_p[0]); mbar_inval(&bar_p[1]);
    for (int i = 0; i < WS_STAGES * WS_CONSUMERS; ++i) { mbar_inval(&bar_full[i]); mbar_inval(&bar_empty[i]); }
  }
  if (warp >= WS_CONSUMERS) return;
  if (NSPLIT > 1) {
    // column-split ranks: accumulators (and, from split 0, the per-sample scalars) go to global memory;
    // cholesky_kernel finishes the job
    const int gid = lane >> 2, tig = lane & 3;
    const int64_t row = s0 + warp * SPW + gid;
    double* grow = args.gram + ((int64_t)q * args.gram_rows + row) * G::NCOL + tile0 * 8 + tig * 2;
#pragma unroll
    for (int ni = 0; ni < NT; ++ni) *reinterpret_cast<double2*>(grow + ni * 8) = make_double2(acc[ni][0], acc[ni][1]);
    if (split == 0 && lane < SPW) {
      double* qd = args.qld + ((int64_t)q * args.gram_rows + s0 + warp * SPW + lane) * 2;
      qd[0] = s_q[warp * SPW + lane]; qd[1] = s_ld[warp * SPW + lane];
    }
    return;
  }
  stage_and_factor<K, NT, CSTR>(acc, Cs, s_q, s_ld, warp * SPW, lane, meta, args, q, s0);
}

// grid = (sample tiles, quasars, column splits)
template <int K, int NL, int MODE, int NSPLIT>
__global__ void __launch_bounds__(WS_THREADS, 1) dla_loglik_ws_kernel(LoglikArgs args) {
  ws_tile<K, NL, MODE, NSPLIT>(args, (int)blockIdx.y + args.q_offset);
}
// The same for the quasars listed in args.only_list = {count, q_0, q_1, ...}: grid.y slots stride over the list (a
// separate kernel: the loop around the tile costs the compiler 500 bytes of spills, which the main kernel must not pay)
template <int K, int NL, int MODE, int NSPLIT>
__global__ void __launch_bounds__(WS_THREADS, 1) dla_loglik_ws_list_kernel(LoglikArgs args) {
  const int nlist = args.only_list[0];
  for (int qi = blockIdx.y; qi < nlist; qi += gridDim.y) {
    ws_tile<K, NL, MODE, NSPLIT>(args, args.only_list[1 + qi]);
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------
// K3 for column-split ranks: Cholesky of B = I + C per sample straight from the global staging rows
// (log_mvnpdf_low_rank.m:22-32), staged through shared memory as an augmented triangle.  Four lanes per
// sample; each lane keeps its columns of the current row in registers (k = 40: 21 kFLOP per sample).
struct CholArgs {
  const QuasarMeta* meta;
  double* gram;                     // [Q x rows x NCOL]
  const double* qld;                // [Q x rows x 2]
  int64_t gram_rows;
  int64_t S;
  double* sample_log_likelihoods;
  int64_t sll_stride;
  double* log_likelihoods_no_dla;   // nullable
  const int32_t* active;
  const int32_t* order;             // tile position -> sample index (see LoglikArgs)
  int q_offset;
};

constexpr int CHOL_SAMPLES = 16;              // samples per CTA of cholesky_kernel
constexpr int CHOL_LANES = 8;                 // lanes per sample
constexpr int CHOL_THREADS = CHOL_SAMPLES * CHOL_LANES;
template <int K>
constexpr size_t cholesky_smem_bytes() { return (size_t)((K + 1) * (K + 2) / 2) * CHOL_SAMPLES * 8; }
// Staging: entry (p, q) of sample s at Cs[chol_slot(aug_index(p, q), s)] -- 16 samples per entry, no padding (k = 40:
// 110 KB, two CTAs per SM), the sample position rotated by 2 * (entry mod 8): the 8 lanes of a sample read 8
// consecutive entries and a half-warp holds two samples, which then fall into 16 different 8-byte bank pairs.
__device__ __forceinline__ int chol_slot(int entry, int s) { return entry * CHOL_SAMPLES + ((s + 2 * (entry & 7)) & (CHOL_SAMPLES - 1)); }

// Left-looking Cholesky, TWO rows (p, p + 1) per step: lane l of a sample owns the columns p + l + 8 j of both rows, so
// every entry of a finished row r that it loads updates two accumulators (loads per FMA halved; the kernel is bound by
// shared-memory loads).  Round 1's version (4 lanes per sample, one row per step, 138 KB per CTA: 64 threads per SM)
// took 12.4 ms per 37 quasars x 10^4 samples at k = 40, three times the Gram itself on the INT8 path.
template <int K>
__global__ void __launch_bounds__(CHOL_THREADS) cholesky_kernel(CholArgs a) {
  using G = GramShape<K>;
  static_assert(K % 2 == 0, "rows are processed in pairs");
  constexpr int NQ = (K + 1 + CHOL_LANES - 1) / CHOL_LANES;      // columns per lane, upper bound
  const int q = (int)blockIdx.y + a.q_offset;
  const QuasarMeta meta = a.meta[q];
  if (meta.nchunks == 0 || (a.active != nullptr && a.active[q] == 0)) return;   // NaNs already written
  extern __shared__ __align__(16) double Cs[];
  const int tid = threadIdx.x, l8 = tid & (CHOL_LANES - 1), sl = tid / CHOL_LANES;
  const int64_t row0 = (int64_t)blockIdx.x * CHOL_SAMPLES;
  // stage the accumulator rows: coalesced along columns, scattered into the augmented triangle
  const double* g0 = a.gram + ((int64_t)q * a.gram_rows + row0) * G::NCOL;
  for (int c = tid; c < G::NCOL; c += CHOL_THREADS) {   // one (divergent) table lookup per column
    const int idx = stage_index_table<K>()[c];
    if (idx >= 0) {
#pragma unroll 8
      for (int r = 0; r < CHOL_SAMPLES; ++r) Cs[chol_slot(idx, r)] = g0[(int64_t)r * G::NCOL + c];
    }
  }
  __syncthreads();
  const unsigned gmask = 0xffu << ((tid & 31) & ~(CHOL_LANES - 1));   // the lanes of this sample
  const int lane0 = (tid & 31) & ~(CHOL_LANES - 1);
  double prod[4] = {1.0, 1.0, 1.0, 1.0};
  for (int p = 0; p < K; p += 2) {
    const int base_p = aug_index<K>(p, p) - p, base_p1 = aug_index<K>(p + 1, p + 1) - (p + 1);   // entry (p, x) at base_p + x
    double v0[NQ], v1[NQ];
#pragma unroll
    for (int j = 0; j < NQ; ++j) {
      const int qq = p + l8 + CHOL_LANES * j;
      v0[j] = (qq <= K) ? Cs[chol_slot(base_p + qq, sl)] : 0.0;
      v1[j] = (qq <= K && qq >= p + 1) ? Cs[chol_slot(base_p1 + qq, sl)] : 0.0;
    }
    if (l8 == 0) v0[0] += 1.0;                                                     // B = I + C   (:23)
    if (l8 == 1) v1[0] += 1.0;
    // finished rows r < p.  The 8 j-entries of a lane are 8 entries apart, so they share one rotated sample slot: one
    // address per (lane, r) and immediate offsets; entry (r, x) sits at base_r + x with base_(r+1) = base_r + K - r
    const int nj = (K - p - l8) / CHOL_LANES + 1;      // columns p + l8 + 8 j <= K
    int base_r = 0;
#pragma unroll 2
    for (int r = 0; r < p; ++r) {
      const int ec = base_r + p, ex = ec + l8;
      const double c0 = Cs[chol_slot(ec, sl)], c1 = Cs[chol_slot(ec + 1, sl)];
      const double* px = Cs + chol_slot(ex, sl);
#pragma unroll
      for (int j = 0; j < NQ; ++j) {
        if (j < nj) {
          const double x = px[j * CHOL_LANES * CHOL_SAMPLES];
          v0[j] = fma(-c0, x, v0[j]);
          v1[j] = fma(-c1, x, v1[j]);
        }
      }
      base_r += K - r;
    }
    // row p: pivot at lane 0, then its entry (p, p + 1) (lane 1) updates row p + 1
    const double d0 = __shfl_sync(gmask, v0[0], lane0);
    prod[(p >> 1) & 1] *= d0;
    const double i0 = rsqrt(d0);
#pragma unroll
    for (int j = 0; j < NQ; ++j) v0[j] *= i0;
    const double c01 = __shfl_sync(gmask, v0[0], lane0 + 1);
#pragma unroll
    for (int j = 0; j < NQ; ++j) v1[j] = fma(-c01, v0[j], v1[j]);
    const double d1 = __shfl_sync(gmask, v1[0], lane0 + 1);
    prod[2 + ((p >> 1) & 1)] *= d1;
    const double i1 = rsqrt(d1);
#pragma unroll
    for (int j = 0; j < NQ; ++j) {
      const int qq = p + l8 + CHOL_LANES * j;
      if (qq <= K && qq > p) Cs[chol_slot(base_p + qq, sl)] = v0[j];
      if (qq <= K && qq > p + 1) Cs[chol_slot(base_p1 + qq, sl)] = v1[j] * i1;
    }
    __syncwarp();
  }
  double zsum = 0.0;
  for (int p = l8; p < K; p += CHOL_LANES) { const double zp = Cs[chol_slot(aug_index<K>(p, K), sl)]; zsum = fma(zp, zp, zsum); }
#pragma unroll
  for (int o = CHOL_LANES / 2; o > 0; o >>= 1) zsum += __shfl_xor_sync(gmask, zsum, o);
  const int64_t row = row0 + sl;
  if (l8 == 0) {
    const double* qd = a.qld + ((int64_t)q * a.gram_rows + row) * 2;
    const double quad = qd[0] - zsum;                                            // :28
    const double logdet = qd[1] + (log(prod[0]) + log(prod[1])) + (log(prod[2]) + log(prod[3]));   // :30
    const double lp = -0.5 * (quad + logdet + (double)meta.n * LOG_2PI);         // :32
    if (row < a.S) a.sample_log_likelihoods[(int64_t)q * a.sll_stride + (a.order ? (int64_t)a.order[row] : row)] = lp;
    else if (row == a.S && a.log_likelihoods_no_dla) a.log_likelihoods_no_dla[q] = lp;
  }
}

// ------------------------------------------------------------------------------------------
// K4: evidence, posteriors, MAP.  One CTA per quasar.
struct EvidenceArgs {
  const QuasarMeta* meta;
  const double* sample_log_likelihoods;   // [Q x S]
  const double* log_likelihoods_no_dla;   // [Q]
  const double* offset_samples;
  const double* log_nhi_samples;
  int64_t S;
  // outputs, each [Q] unless noted
  double *min_z_dlas, *max_z_dlas, *log_priors_no_dla, *log_priors_dla, *log_likelihoods_dla, *log_posteriors_no_dla,
      *log_posteriors_dla, *model_posteriors /*[Q x 2]*/, *p_no_dlas, *p_dlas, *map_z_dlas, *map_log_nhis;
  int64_t* map_inds;
};

__global__ void __launch_bounds__(NTHREADS) evidence_kernel(EvidenceArgs a) {
  const int q = blockIdx.x, tid = threadIdx.x;
  const QuasarMeta meta = a.meta[q];
  const double* ll = a.sample_log_likelihoods + (int64_t)q * a.S;
  __shared__ double s_val[NTHREADS / 32];
  __shared__ long long s_idx[NTHREADS / 32];
  __shared__ double s_max;
  __shared__ long long s_arg;
  __shared__ int s_nan;

  // max over samples, NaN-ignoring like MATLAB max (process_qsos.m:203); first index attaining it
  double m = -INFINITY; long long arg = -1; int has_nan = 0;
  for (int64_t s = tid; s < a.S; s += NTHREADS) {
    double v = ll[s];
    if (v != v) { has_nan = 1; continue; }
    if (v > m || arg < 0) { m = v; arg = s; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    double om = __shfl_xor_sync(0xffffffffu, m, o);
    long long oa = __shfl_xor_sync(0xffffffffu, arg, o);
    if (oa >= 0 && (arg < 0 || om > m || (om == m && oa < arg))) { m = om; arg = oa; }
  }
  has_nan = __any_sync(0xffffffffu, has_nan);
  if (tid == 0) s_nan = 0;
  __syncthreads();
  if ((tid & 31) == 0) { s_val[tid >> 5] = m; s_idx[tid >> 5] = arg; if (has_nan) atomicOr(&s_nan, 1); }
  __syncthreads();
  if (tid == 0) {
    for (int w = 1; w < NTHREADS / 32; ++w) {
      double om = s_val[w]; long long oa = s_idx[w];
      if (oa >= 0 && (arg < 0 || om > m || (om == m && oa < arg))) { m = om; arg = oa; }
    }
    s_max = m; s_arg = arg;
  }
  __syncthreads();
  m = s_max; arg = s_arg;
  double sum = 0.0;
  for (int64_t s = tid; s < a.S; s += NTHREADS) sum += exp(ll[s] - m);          // :205-207 (NaN propagates like mean)
  sum = warp_sum(sum);
  __syncthreads();
  if ((tid & 31) == 0) s_val[tid >> 5] = sum;
  __syncthreads();
  if (tid == 0) {
    for (int w = 1; w < NTHREADS / 32; ++w) sum += s_val[w];
    const bool valid = meta.nchunks > 0;
    double lldla = valid ? m + log(sum / (double)a.S) : NAN;                     // :209-210
    double llno = a.log_likelihoods_no_dla[q];
    double lpno = meta.log_prior_no_dla + llno;                                  // :153-154
    double lpdla = meta.log_prior_dla + lldla;                                   // :212-213
    a.min_z_dlas[q] = meta.min_z_dla; a.max_z_dlas[q] = meta.max_z_dla;
    a.log_priors_no_dla[q] = meta.log_prior_no_dla; a.log_priors_dla[q] = meta.log_prior_dla;
    a.log_likelihoods_dla[q] = lldla;
    a.log_posteriors_no_dla[q] = valid ? lpno : NAN; a.log_posteriors_dla[q] = valid ? lpdla : NAN;
    // model posteriors (process_qsos.m:224-233); MATLAB max ignores NaN
    double mx = fmax(lpno, lpdla);
    double e0 = exp(lpno - mx), e1 = exp(lpdla - mx);
    double tot = e0 + e1;
    double p0 = e0 / tot, p1 = e1 / tot;
    if (!valid) { p0 = NAN; p1 = NAN; }
    a.model_posteriors[2 * q] = p0; a.model_posteriors[2 * q + 1] = p1;
    a.p_no_dlas[q] = p0; a.p_dlas[q] = 1.0 - p0;
    // MAP (generate_ascii_catalog.m:73-80)
    a.map_inds[q] = (valid && arg >= 0) ? arg : -1;
    if (valid && arg >= 0) {
      a.map_z_dlas[q] = __dadd_rn(meta.min_z_dla, __dmul_rn(meta.max_z_dla - meta.min_z_dla, a.offset_samples[arg]));
      a.map_log_nhis[q] = a.log_nhi_samples[arg];
    } else {
      a.map_z_dlas[q] = NAN; a.map_log_nhis[q] = NAN;
    }
  }
}

// ------------------------------------------------------------------------------------------
// Multi-DLA level post-processing (multi_dlas/process_qsos_multiple_dlas_meanflux.m:359-472).
// One CTA per quasar, after the log-likelihood kernel of a level (or of the sub-DLA pass, level 0):
// Occam term -log S per sample (:361,378), z-separation filter (:386-392), nan-LSE (:400-409,416-426),
// MAP (:438-445), early exit (:460-464), weighted resampling with replacement (:466-472).
struct MultiLevelArgs {
  const QuasarMeta* meta;
  double* sll;                  // this level's sample log-likelihoods, [Q] rows of S with stride sll_stride; in/out
  int64_t sll_stride;
  int64_t S;
  int level;                    // 1..max_dlas; 0 = sub-DLA (LLS) pass
  int max_dlas;
  int32_t* partners;            // [Q x 3 x S] base_sample_inds (0-based), row level-1 written here
  const int32_t* partners_in;   // optional given base_sample_inds [Q x 3 x S] (parity runs); nullptr = resample
  int32_t* active;              // [Q] level loop still running
  const double* offset_samples;
  const double* log_nhi_samples;
  const double* uniforms;       // [3 x S]: rand stream after rng('default'), S numbers per level (:143,471)
  double min_z_separation;      // kms_to_z(3000), :33
  double* cum_scratch;          // [Q x S]
  double* log_likelihoods;      // level >= 1: [Q x max_dlas]; level 0: [Q] (log_likelihoods_lls)
  double* map_z;                // [Q x max_dlas x max_dlas]
  double* map_log_nhi;          // [Q x max_dlas x max_dlas]
  int64_t* map_inds;            // [Q x max_dlas x max_dlas], 0-based, -1 = unset
};

__global__ void __launch_bounds__(NTHREADS) multi_level_kernel(MultiLevelArgs a) {
  const int q = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const QuasarMeta meta = a.meta[q];
  const int64_t S = a.S;
  const int L = a.level, MD = a.max_dlas;
  double* ll = a.sll + (int64_t)q * a.sll_stride;
  __shared__ double s_val[NTHREADS / 32], s_val2[NTHREADS / 32];
  __shared__ long long s_idx[NTHREADS / 32];
  __shared__ double s_max, s_sum, s_cnt, s_ev;
  __shared__ long long s_arg;
  __shared__ double s_scan[NTHREADS];

  if (L >= 1 && tid < MD) {   // this level's MAP row starts unset (:129-131)
    const int64_t o = ((int64_t)q * MD + (L - 1)) * MD + tid;
    a.map_z[o] = NAN; a.map_log_nhi[o] = NAN; a.map_inds[o] = -1;
  }
  const bool live = meta.nchunks > 0 && a.active[q] != 0;
  if (!live) {
    if (tid == 0) {
      if (L >= 1) a.log_likelihoods[(int64_t)q * MD + (L - 1)] = NAN; else a.log_likelihoods[q] = NAN;
    }
    return;
  }
  const double logS = log((double)S);
  const double zmin = meta.min_z_dla, zspan = meta.max_z_dla - meta.min_z_dla;
  const int32_t* part = a.partners + (int64_t)q * 3 * S;
  auto zs = [&](int64_t s) { return __dadd_rn(zmin, __dmul_rn(zspan, a.offset_samples[s])); };

  // ---- pass 1: Occam term, separation filter, nan-max with first index
  double m = -INFINITY; long long arg = -1;
  for (int64_t s = tid; s < S; s += NTHREADS) {
    double v = ll[s] - logS;                                                       // :361 / :378
    if (L >= 2) {                                                                  // :386-392
      double z[4];
      z[0] = zs(s);
      for (int j = 0; j < L - 1; ++j) z[j + 1] = zs(part[(int64_t)j * S + s]);
      for (int i = 1; i < L; ++i) {                                                // insertion sort (<= 4 values)
        double zi = z[i]; int k = i - 1;
        while (k >= 0 && z[k] > zi) { z[k + 1] = z[k]; --k; }
        z[k + 1] = zi;
      }
      bool close = false;
      for (int i = 1; i < L; ++i) close |= (z[i] - z[i - 1]) < a.min_z_separation;
      if (close) v = NAN;
    }
    ll[s] = v;
    if (v == v && (arg < 0 || v > m)) { m = v; arg = s; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    double om = __shfl_xor_sync(0xffffffffu, m, o);
    long long oa = __shfl_xor_sync(0xffffffffu, arg, o);
    if (oa >= 0 && (arg < 0 || om > m || (om == m && oa < arg))) { m = om; arg = oa; }
  }
  if (lane == 0) { s_val[wid] = m; s_idx[wid] = arg; }
  __syncthreads();
  if (tid == 0) {
    for (int w = 1; w < NTHREADS / 32; ++w) {
      double om = s_val[w]; long long oa = s_idx[w];
      if (oa >= 0 && (arg < 0 || om > m || (om == m && oa < arg))) { m = om; arg = oa; }
    }
    s_max = m; s_arg = arg;
  }
  __syncthreads();
  m = s_max; arg = s_arg;

  // ---- pass 2: nan-mean of exp(ll - max)
  double sum = 0.0, cnt = 0.0;
  for (int64_t s = tid; s < S; s += NTHREADS) {
    double v = ll[s];
    if (v == v) { sum += exp(v - m); cnt += 1.0; }
  }
  sum = warp_sum(sum); cnt = warp_sum(cnt);
  __syncthreads();
  if (lane == 0) { s_val[wid] = sum; s_val2[wid] = cnt; }
  __syncthreads();
  if (tid == 0) {
    for (int w = 1; w < NTHREADS / 32; ++w) { sum += s_val[w]; cnt += s_val2[w]; }
    s_sum = sum; s_cnt = cnt;
    double ev = (arg >= 0) ? m + log(sum / cnt) - logS * (double)(L >= 1 ? L - 1 : 0) : NAN;   // :407-409 / :424-426
    s_ev = ev;
    if (L >= 1) a.log_likelihoods[(int64_t)q * MD + (L - 1)] = ev; else a.log_likelihoods[q] = ev;
    if (L >= 1 && arg >= 0) {                                                      // :438-445
      const int64_t o = ((int64_t)q * MD + (L - 1)) * MD;
      a.map_inds[o] = arg; a.map_z[o] = zs(arg); a.map_log_nhi[o] = a.log_nhi_samples[arg];
      for (int j = 0; j < L - 1; ++j) {
        const long long k = part[(int64_t)j * S + arg];
        a.map_inds[o + j + 1] = k; a.map_z[o + j + 1] = zs(k); a.map_log_nhi[o + j + 1] = a.log_nhi_samples[k];
      }
    }
    if (L >= 1 && L < MD && !(ev == ev)) a.active[q] = 0;                          // :460-464
  }
  __syncthreads();
  if (L < 1 || L >= MD || !(s_ev == s_ev)) return;                                 // :452-454, :460-464

  // ---- resampling: base_sample_inds(level, :) = randsample(S, S, true, W)      :466-472
  int32_t* out = a.partners + ((int64_t)q * 3 + (L - 1)) * S;
  if (a.partners_in != nullptr) {
    const int32_t* in = a.partners_in + ((int64_t)q * 3 + (L - 1)) * S;
    for (int64_t s = tid; s < S; s += NTHREADS) out[s] = in[s];
    return;
  }
  const double total = s_sum;
  double* cum = a.cum_scratch + (int64_t)q * S;
  const int64_t seg = (S + NTHREADS - 1) / NTHREADS;
  const int64_t b = min((int64_t)tid * seg, S), e = min(b + seg, S);
  double local = 0.0;
  for (int64_t s = b; s < e; ++s) {
    double v = ll[s];
    local += (v == v) ? exp(v - m) / total : 0.0;                                  // W(nanind) = 0; p = w / sum(w)
  }
  s_scan[tid] = local;
  __syncthreads();
  if (tid == 0) {
    double run = 0.0;
    for (int t = 0; t < NTHREADS; ++t) { double x = s_scan[t]; s_scan[t] = run; run += x; }
  }
  __syncthreads();
  double run = s_scan[tid];
  for (int64_t s = b; s < e; ++s) {
    double v = ll[s];
    run += (v == v) ? exp(v - m) / total : 0.0;
    cum[s] = fmin(run, 1.0);                                                       // edges = min([0 cumsum(p)], 1)
  }
  __syncthreads();
  const double* u = a.uniforms + (int64_t)(L - 1) * S;
  for (int64_t t = tid; t < S; t += NTHREADS) {
    const double x = u[t];
    int64_t lo = 0, hi = S - 1;            // number of interior edges cum[0..S-2] that are <= x
    while (lo < hi) {
      int64_t mid = (lo + hi) >> 1;
      if (cum[mid] <= x) lo = mid + 1; else hi = mid;
    }
    out[t] = (int32_t)lo;
  }
}

// Multi-DLA priors and model posteriors (...meanflux.m:190-216, 300-301, 411-413, 428-430, 482-495).
struct MultiPosteriorArgs {
  const QuasarMeta* meta;
  int64_t Q;
  int max_dlas;
  double Z_lls, Z_dla;
  const double* log_likelihoods_no_dla;   // [Q]
  const double* log_likelihoods_lls;      // [Q]
  const double* log_likelihoods_dla;      // [Q x max_dlas]
  double *min_z_dlas, *max_z_dlas, *log_priors_no_dla, *log_priors_lls, *log_priors_dla /*[Q x max_dlas]*/;
  double *log_posteriors_no_dla, *log_posteriors_lls, *log_posteriors_dla /*[Q x max_dlas]*/;
  double *model_posteriors /*[Q x (2 + max_dlas)]*/, *p_no_dlas, *p_lls, *p_dlas;
};

__global__ void multi_posterior_kernel(MultiPosteriorArgs a) {
  const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= a.Q) return;
  const QuasarMeta meta = a.meta[q];
  const int MD = a.max_dlas;
  const double nq = (double)meta.prior_num_quasars, nd = (double)meta.prior_num_dlas;
  double pd[8];
  const double p1 = nd / nq;
  for (int j = 0; j < MD; ++j) pd[j] = pow(p1, (double)(j + 1));                   // :194
  for (int j = 0; j < MD - 1; ++j) pd[j] = pd[j] - pd[j + 1];                      // :197-199
  const double lp_lls_prior = log(nd) - log(nq) + log(a.Z_lls) - log(a.Z_dla);    // :208-210
  const double lp_no_prior = log(nq - nd - a.Z_lls * nd / a.Z_dla) - log(nq);     // :214-216
  a.min_z_dlas[q] = meta.min_z_dla; a.max_z_dlas[q] = meta.max_z_dla;
  a.log_priors_no_dla[q] = lp_no_prior; a.log_priors_lls[q] = lp_lls_prior;
  double lp[10];
  lp[0] = lp_no_prior + a.log_likelihoods_no_dla[q];                               // :300-301
  lp[1] = lp_lls_prior + a.log_likelihoods_lls[q];                                 // :428-430
  for (int j = 0; j < MD; ++j) {
    const double pr = log(pd[j]);                                                  // :204
    a.log_priors_dla[q * MD + j] = pr;
    lp[2 + j] = pr + a.log_likelihoods_dla[q * MD + j];                            // :411-413
    a.log_posteriors_dla[q * MD + j] = lp[2 + j];
  }
  a.log_posteriors_no_dla[q] = lp[0]; a.log_posteriors_lls[q] = lp[1];
  double mx = -INFINITY; bool any = false;
  for (int j = 0; j < MD + 2; ++j) if (lp[j] == lp[j]) { mx = any ? fmax(mx, lp[j]) : lp[j]; any = true; }   // max ignores NaN
  if (!any) mx = NAN;
  double e[10], tot = 0.0;
  for (int j = 0; j < MD + 2; ++j) { e[j] = exp(lp[j] - mx); tot += e[j]; }        // :485-488; sum propagates NaN
  const double inv = 1.0 / tot;                                                    // :490-491
  for (int j = 0; j < MD + 2; ++j) a.model_posteriors[q * (MD + 2) + j] = e[j] * inv;
  const double p_no = e[0] * inv, p_l = e[1] * inv;
  a.p_no_dlas[q] = p_no; a.p_lls[q] = p_l; a.p_dlas[q] = 1.0 - p_no - p_l;          // :493-495
}

}  // namespace gpdla
