// Draws from the learned model on the device: mock spectra from the prior predictive of the single- or multi-DLA
// model, or absorbers injected into given spectra, with the truth of every draw (see gpdla_draw_spectra in gpdla.h).
// The pieces are the ones the inference evaluates: the window scan and priors of prepare_quasars_kernel
// (scan_window, dla_z_range, single_dla_log_priors, multi_dla_log_priors), the absorption of reconstruct_kernel
// (window_absorption) and the per-pixel null model (null_model_pixel).  Random numbers are counter-based
// (Philox4x32-10), so a draw depends on (seed, quasar index in the catalogue, stream, element) only.
// One CTA per quasar; no atomics and no cross-thread floating-point sums: repeated calls give the same bits.
#pragma once
#include <stdint.h>
#include "gpdla_reconstruct.cuh"

namespace gpdla {

constexpr int DRAW_MAX_ABSORBERS = 4;
constexpr int DRAW_MAX_ATTEMPTS = 64;      // redraws of a j-DLA set until its redshifts are separated
// the four random streams of one quasar (counter word 1)
constexpr uint32_t RNG_MODEL = 0, RNG_INDEX = 1, RNG_LATENT = 2, RNG_PIXEL = 3;

// Philox4x32-10 (Salmon et al. 2011): the bits of curand's curand_Philox4x32_10 for the same counter and key
__host__ __device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    if (r > 0) { k.x += 0x9E3779B9u; k.y += 0xBB67AE85u; }
#ifdef __CUDA_ARCH__
    const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), hi1 = __umulhi(0xCD9E8D57u, c.z);
#else
    const uint32_t hi0 = (uint32_t)(((uint64_t)0xD2511F53u * c.x) >> 32),
                   hi1 = (uint32_t)(((uint64_t)0xCD9E8D57u * c.z) >> 32);
#endif
    const uint32_t lo0 = 0xD2511F53u * c.x, lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
  }
  return c;
}

// The two 64-bit words of one draw: counter (element, stream, g_lo, g_hi), key = seed.  W0 = r.y:r.x, W1 = r.w:r.z.
__device__ __forceinline__ void draw_words(uint64_t seed, uint64_t g, uint32_t stream, uint32_t element, uint64_t& w0,
                                           uint64_t& w1) {
  const uint4 r = philox4x32_10(make_uint4(element, stream, (uint32_t)g, (uint32_t)(g >> 32)),
                                make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
  w0 = ((uint64_t)r.y << 32) | r.x;
  w1 = ((uint64_t)r.w << 32) | r.z;
}
// ((W >> 11) + 0.5) 2^-53: a uniform in (0, 1) (the largest word rounds to 1)
__device__ __forceinline__ double word_uniform(uint64_t w) { return ((double)(w >> 11) + 0.5) * 0x1p-53; }
// Box-Muller on the uniforms of the two words
__device__ __forceinline__ void word_normals(uint64_t w0, uint64_t w1, double& n0, double& n1) {
  const double r = sqrt(-2.0 * log(word_uniform(w0))), t = 2.0 * word_uniform(w1);
  n0 = r * cospi(t);
  n1 = r * sinpi(t);
}

struct DrawArgs {
  // spectra, padded [Q x L_max]; flux_in is read only when injecting
  const double* wavelengths;
  const double* flux_in;
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
  int n_rest;
  double c_0, tau_0, beta;
  double min_lambda, max_lambda, lya_wavelength, lyman_limit, prior_z_qso_increase, min_z_cut, max_z_cut,
      pixel_spacing;
  int num_lines;
  // model 0: single-DLA (null model with s = 1); model 1: multi-DLA (mean-flux null model)
  int model, max_dlas;
  int inject, from_prior;
  uint64_t seed;
  int64_t first_quasar;
  // prior source: prior catalogue, samples (caller's order), sub-DLA samples and normalisers
  const double* prior_z_qsos;
  const uint8_t* prior_dla_ind;
  int64_t n_prior;
  const double* offset_samples;
  const double* log_nhi_samples;
  const double* nhi_samples;
  const double* lls_nhi_samples;
  int64_t S;
  double Z_lls, Z_dla, min_z_separation;
  // given source: [Q x num_absorbers], NaN z = none
  int num_absorbers;
  const double* absorber_z;
  const double* absorber_nhi;
  // outputs: flux and absorption [Q x L_max] (absorption nullable); truth [Q] and [Q x truth_width] (prior source)
  double* flux;
  double* absorption;
  int32_t* truth_model;
  int64_t* truth_inds;
  double* truth_z;
  double* truth_log_nhi;
  int truth_width;
};

template <int K>
__host__ __device__ constexpr size_t draw_smem_doubles(int64_t L_max) {
  return (size_t)L_max + (NTHREADS + 6) + MAX_LINES + K;   // s_a, s_raw, s_mult, s_xi
}

template <int K>
__global__ void __launch_bounds__(NTHREADS) draw_spectra_kernel(const __grid_constant__ DrawArgs a) {
  static_assert(K % 2 == 0, "latent normals come in pairs");
  const int q = blockIdx.x, tid = threadIdx.x;
  const int64_t L_max = a.L_max;
  const int64_t L = min(max((int64_t)a.lengths[q], (int64_t)0), L_max);
  const double z_qso = a.z_qsos[q];
  const double* wl = a.wavelengths + q * L_max;
  const double* nv = a.noise_variance + q * L_max;
  const uint8_t* pmask = a.pixel_mask + q * L_max;
  const double* fin = a.inject ? a.flux_in + q * L_max : nullptr;
  const uint64_t g = (uint64_t)(a.first_quasar + q);

  extern __shared__ __align__(16) double dr_smem[];
  double* s_a = dr_smem;
  double* s_raw = s_a + L_max;
  double* s_mult = s_raw + NTHREADS + 6;
  double* s_xi = s_mult + MAX_LINES;
  __shared__ double s_abz[DRAW_MAX_ABSORBERS], s_abn[DRAW_MAX_ABSORBERS];
  // thread 0's working set of the prior draw (shared, so that its dynamic indexing needs no stack frame)
  __shared__ double s_p[2 + DRAW_MAX_ABSORBERS], s_tz[DRAW_MAX_ABSORBERS], s_tn[DRAW_MAX_ABSORBERS];
  __shared__ int64_t s_ind[DRAW_MAX_ABSORBERS];
  __shared__ int s_num, s_code;

  const WindowScan ws = scan_window(wl, pmask, L, z_qso, a.min_lambda, a.max_lambda, a.prior_z_qsos, a.prior_dla_ind,
                                    a.from_prior ? a.n_prior : 0, a.prior_z_qso_increase);

  // the absorbers: given, or one draw from the model prior (one thread)
  if (tid == 0) {
    int code = 0, num = 0;
    if (!a.from_prior) {
      num = a.num_absorbers;
      for (int b = 0; b < num; ++b) {
        s_abz[b] = a.absorber_z[(int64_t)q * num + b];
        s_abn[b] = a.absorber_nhi[(int64_t)q * num + b];
      }
    } else {
      const int TW = a.truth_width;
      int64_t* ind = s_ind;
      double *tz = s_tz, *tn = s_tn, *p = s_p;
      double min_z, max_z;
      dla_z_range(ws.minw, ws.maxw, z_qso, a.lya_wavelength, a.lyman_limit, a.min_z_cut, a.max_z_cut, min_z, max_z);
      // model probabilities in the order of the truth codes: single {none, 1 DLA}, multi {none, sub-DLA, 1..J DLAs}
      int nm;
      if (a.model == 0) {
        single_dla_log_priors(ws.prior_num_quasars, ws.prior_num_dlas, p[0], p[1]);
        nm = 2;
      } else {
        multi_dla_log_priors(ws.prior_num_quasars, ws.prior_num_dlas, a.Z_lls, a.Z_dla, a.max_dlas, p[0], p[1], p + 2);
        nm = 2 + a.max_dlas;
      }
      bool finite = ws.n > 0;
      for (int m = 0; m < nm; ++m) { p[m] = exp(p[m]); finite = finite && isfinite(p[m]); }
      if (!finite) {
        code = -1;
      } else {
        uint64_t w0, w1;
        draw_words(a.seed, g, RNG_MODEL, 0, w0, w1);
        const double u = word_uniform(w0);
        int m = nm - 1;
        double cum = 0.0;
        for (int t = 0; t < nm; ++t) {
          cum += p[t];
          if (u < cum) { m = t; break; }
        }
        code = (a.model == 0 && m == 1) ? 2 : m;        // 0 none, 1 sub-DLA, 1 + j: j DLAs
        const int j = code >= 2 ? code - 1 : code;      // absorbers to place
        const double span = max_z - min_z;
        bool placed = j == 0;
        for (int att = 0; att < DRAW_MAX_ATTEMPTS && !placed; ++att) {
          for (int s = 0; s < j; ++s) {
            draw_words(a.seed, g, RNG_INDEX, (uint32_t)(4 * att + s), w0, w1);
            const int64_t i = (int64_t)__umul64hi(w0, (uint64_t)a.S);
            int k = s - 1;                              // insertion in ascending z (as multi_level_kernel's filter)
            const double z = __dadd_rn(min_z, __dmul_rn(span, a.offset_samples[i]));
            while (k >= 0 && tz[k] > z) { tz[k + 1] = tz[k]; ind[k + 1] = ind[k]; --k; }
            tz[k + 1] = z; ind[k + 1] = i;
          }
          bool close = false;
          for (int s = 1; s < j; ++s) close |= (tz[s] - tz[s - 1]) < a.min_z_separation;
          placed = !close;
        }
        if (!placed) {
          code = -2;
        } else {
          num = j;
          for (int s = 0; s < j; ++s) {
            const double N = code == 1 ? a.lls_nhi_samples[ind[s]] : a.nhi_samples[ind[s]];
            s_abz[s] = tz[s]; s_abn[s] = N;
            tn[s] = code == 1 ? log10(N) : a.log_nhi_samples[ind[s]];
          }
        }
      }
      a.truth_model[q] = code;
      for (int s = 0; s < TW; ++s) {
        const bool on = code > 0 && s < num;
        a.truth_inds[(int64_t)q * TW + s] = on ? ind[s] : -1;
        a.truth_z[(int64_t)q * TW + s] = on ? tz[s] : NAN;
        a.truth_log_nhi[(int64_t)q * TW + s] = on ? tn[s] : NAN;
      }
    }
    s_num = num; s_code = code;
  }
  __syncthreads();

  if (ws.n == 0 || s_code < 0) {   // nothing modelled, or no draw: a NaN row
    for (int64_t i = tid; i < L_max; i += NTHREADS) {
      a.flux[q * L_max + i] = NAN;
      if (a.absorption) a.absorption[q * L_max + i] = NAN;
    }
    return;
  }
  const int first = ws.first, n_u = ws.n_u;
  window_absorption(s_a, s_raw, s_mult, n_u, wl + first, log10(ws.minu), log10(ws.maxu), a.pixel_spacing, a.num_lines,
                    s_num, s_abz, s_abn);
  if (!a.inject) {
    for (int c = tid; c < K / 2; c += NTHREADS) {
      uint64_t w0, w1;
      draw_words(a.seed, g, RNG_LATENT, (uint32_t)c, w0, w1);
      word_normals(w0, w1, s_xi[2 * c], s_xi[2 * c + 1]);
    }
    __syncthreads();
  }

  for (int64_t i = tid; i < L_max; i += NTHREADS) {
    double y, ab = NAN;
    if (i >= L) {
      y = a.inject ? fin[i] : 0.0;                                  // the padding of pad_spectra
    } else {
      const double w = wl[i], rest = w / (1.0 + z_qso);
      if (!(rest >= a.min_lambda && rest <= a.max_lambda)) {
        y = a.inject ? fin[i] : NAN;                                // outside the modelled window
      } else {
        ab = s_a[i - first];
        uint64_t w0, w1;
        draw_words(a.seed, g, RNG_PIXEL, (uint32_t)i, w0, w1);
        double e1, e2;
        word_normals(w0, w1, e1, e2);
        if (a.inject) {
          const double ex = 1.0 - ab * ab;                          // the noise variance stays v
          y = ab * fin[i] + (ex > 0.0 ? sqrt(ex * nv[i]) * e2 : 0.0);
        } else {
          const PixelModel m = null_model_pixel(a.rest_wavelengths, a.mu, a.log_omega, a.n_rest, a.c_0, a.tau_0,
                                                a.beta, a.lya_wavelength, a.model, w, rest, z_qso);
          double mx = 0.0;
#pragma unroll
          for (int c = 0; c < K; ++c) mx = fma(interp_linear(a.rest_wavelengths, a.M + c, K, m.j, rest), s_xi[c], mx);
          y = ab * (m.mu * m.absorb + m.absorb * mx + sqrt(m.om2) * e1) + sqrt(nv[i]) * e2;
        }
      }
    }
    a.flux[q * L_max + i] = y;
    if (a.absorption) a.absorption[q * L_max + i] = ab;
  }
}

}  // namespace gpdla
