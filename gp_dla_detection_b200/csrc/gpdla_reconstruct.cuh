// The fitted model of each quasar under a chosen list of absorbers: the GP-conditional continuum, the model mean and
// standard deviation on the quasar's own pixel grid, and the Gaussian log-density at that one parameter point.  What the
// reference draws on the host in CDDF_analysis/qso_loader.py:1654-1774 (plot_this_mu), evaluated with the hot path's
// own pieces: the per-pixel null model of prepare_quasars_kernel (null_model_pixel), the padded grid, and the
// absorption of voigt_batch_kernel (direct line sum, exp_nonpos, 7-tap instrument profile).
//
// Per quasar, over the used pixels (window and not masked), with a = product of the convolved absorber profiles:
//   d = a^2 om2~ + v,  r = y - a mu~,  B = I + (a M~)' D^-1 (a M~),  g = (a M~)' D^-1 r,  x^ = B^-1 g
//   chi2 = sum r^2/d - g' B^-1 g,  log p = -1/2 (chi2 + sum log d + log det B + n log 2pi)
// One CTA per quasar; every sum has a fixed owner and a fixed order, no atomics.
#pragma once
#include <stdint.h>
#include "gpdla_kernels.cuh"

namespace gpdla {

constexpr int RC_CHUNK = 128;       // pixels per staged chunk of (a M~ | r) rows
constexpr int RC_MAX_ABSORBERS = 4;

struct ReconArgs {
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
  int n_rest;
  double c_0, tau_0, beta;
  double min_lambda, max_lambda, lya_wavelength, pixel_spacing;
  int num_lines;
  int meanflux;
  // absorbers [Q x num_absorbers]; NaN z = no absorber
  int num_absorbers;
  const double* absorber_z;
  const double* absorber_nhi;
  // outputs, each nullable: planes [Q x L_max], latent [Q x k], scalars [Q]
  double *absorption, *prior_mean, *prior_sd, *fit_mean, *continuum, *continuum_sd;
  double *latent, *chi2, *log_likelihood;
  int32_t* num_pixels;
};

// The absorption of one quasar's window on the padded grid (process_qsos.m:168-188; ...meanflux.m:342-351): each
// absorber's profile as voigt_batch_kernel computes it (num_lines lines, direct optical depth, exp_nonpos, 7-tap
// instrument profile), the convolved profiles multiplied in the given order into s_a[0, n_u).  Absorber b is
// (abs_z[b], abs_nhi[b]); a NaN z is no absorber.  s_raw holds NTHREADS + 6 doubles, s_mult MAX_LINES.  All NTHREADS
// threads call it; s_a is complete when it returns.  reconstruct_kernel and draw_spectra_kernel both build it here.
__device__ __forceinline__ void window_absorption(double* s_a, double* s_raw, double* s_mult, int n_u,
                                                  const double* wl_first, double lo, double hi, double pixel_spacing,
                                                  int num_lines, int num_absorbers, const double* abs_z,
                                                  const double* abs_nhi) {
  const int tid = threadIdx.x;
  for (int i = tid; i < n_u; i += NTHREADS) s_a[i] = 1.0;
  for (int b = 0; b < num_absorbers; ++b) {
    const double z = abs_z[b];
    if (z != z) continue;   // NaN: no absorber in this slot
    const double N = abs_nhi[b];
    __syncthreads();
    if (tid < num_lines) s_mult[tid] = line_multiplier(tid, z);
    for (int i0 = 0; i0 < n_u; i0 += NTHREADS) {
      __syncthreads();
      for (int t = tid; t < NTHREADS + 6; t += NTHREADS) {
        const int p = i0 + t;
        if (p < n_u + 6) {
          const double tau = tau_sum_generic(padded_wavelength(p, n_u, wl_first, lo, hi, pixel_spacing), s_mult, 1,
                                             num_lines);
          s_raw[t] = exp_nonpos(-N * tau);                              // voigt.c:291
        }
      }
      __syncthreads();
      const int i = i0 + tid;
      if (i < n_u) {
        double acc = 0.0;
#pragma unroll
        for (int t = 0; t < 7; ++t) acc = fma(s_raw[tid + t], c_lines.ip[t], acc);   // voigt.c:297-299
        s_a[i] = s_a[i] * acc;
      }
    }
  }
  __syncthreads();
}

// dynamic shared memory of reconstruct_kernel<K> for rows of L_max pixels
template <int K>
__host__ __device__ constexpr size_t reconstruct_smem_doubles(int64_t L_max) {
  return (size_t)L_max                          // s_a: absorption of the window pixels
         + (NTHREADS + 6)                       // s_raw: raw profile chunk
         + MAX_LINES                            // s_mult
         + (size_t)RC_CHUNK * (K + 1)           // s_u: staged (a M~ | r) rows
         + 2 * RC_CHUNK                         // s_dinv, s_logd
         + (size_t)K * (K + 1)                  // s_L: B, then its Cholesky factor (lower)
         + 3 * K;                               // s_y, s_x, s_rdiag
}

template <int K>
__global__ void __launch_bounds__(NTHREADS) reconstruct_kernel(const __grid_constant__ ReconArgs a) {
  constexpr int KA = K + 1;                                  // augmented column: r
  constexpr int NAUG = (K + 1) * (K + 2) / 2;                // entries (p <= q <= K) of the augmented Gram
  constexpr int NE = (NAUG + 1 + NTHREADS - 1) / NTHREADS;  // entries per thread (+1: sum log d)
  const int q = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t L_max = a.L_max;
  const int64_t L = min(max((int64_t)a.lengths[q], (int64_t)0), L_max);
  const double z_qso = a.z_qsos[q];
  const double* wl = a.wavelengths + q * L_max;
  const double* fl = a.flux + q * L_max;
  const double* nv = a.noise_variance + q * L_max;
  const uint8_t* pmask = a.pixel_mask + q * L_max;

  extern __shared__ __align__(16) double rc_smem[];
  double* s_a = rc_smem;
  double* s_raw = s_a + L_max;
  double* s_mult = s_raw + NTHREADS + 6;
  double* s_u = s_mult + MAX_LINES;
  double* s_dinv = s_u + RC_CHUNK * KA;
  double* s_logd = s_dinv + RC_CHUNK;
  double* s_L = s_logd + RC_CHUNK;            // [K][K + 1]
  double* s_y = s_L + K * KA;
  double* s_x = s_y + K;
  double* s_rdiag = s_x + K;
  __shared__ int r_first[NTHREADS / 32], r_last[NTHREADS / 32], r_n[NTHREADS / 32];
  __shared__ double r_min[NTHREADS / 32], r_max[NTHREADS / 32];
  __shared__ int s_first, s_nu, s_n;
  __shared__ double s_lo, s_hi, s_aug[NAUG + 1];

  // window / mask (process_qsos.m:102-110): first and last window pixel, used count, extreme window wavelengths
  {
    int first = 1 << 30, last = -1, n = 0;
    double minu = INFINITY, maxu = -INFINITY;
    for (int64_t i = tid; i < L; i += NTHREADS) {
      const double w = wl[i], rest = w / (1.0 + z_qso);
      if (rest >= a.min_lambda && rest <= a.max_lambda) {
        first = min(first, (int)i); last = max(last, (int)i);
        minu = fmin(minu, w); maxu = fmax(maxu, w);
        n += !pmask[i];
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      first = min(first, __shfl_xor_sync(0xffffffffu, first, o));
      last = max(last, __shfl_xor_sync(0xffffffffu, last, o));
      n += __shfl_xor_sync(0xffffffffu, n, o);
      minu = fmin(minu, __shfl_xor_sync(0xffffffffu, minu, o));
      maxu = fmax(maxu, __shfl_xor_sync(0xffffffffu, maxu, o));
    }
    if (lane == 0) { r_first[warp] = first; r_last[warp] = last; r_n[warp] = n; r_min[warp] = minu; r_max[warp] = maxu; }
    __syncthreads();
    if (tid == 0) {
      for (int w = 1; w < NTHREADS / 32; ++w) {
        first = min(first, r_first[w]); last = max(last, r_last[w]); n += r_n[w];
        minu = fmin(minu, r_min[w]); maxu = fmax(maxu, r_max[w]);
      }
      // warp 0's values are already in first/last/n/minu/maxu; the other warps' are added in warp order
      s_first = first; s_nu = last >= first ? last - first + 1 : 0; s_n = n;
      s_lo = log10(minu); s_hi = log10(maxu);
    }
    __syncthreads();
  }
  const int first = s_first, n_u = s_nu, n_used = s_n;

  if (n_used == 0) {   // process_qsos.m:74-82: nothing to condition on
    for (int64_t i = tid; i < L_max; i += NTHREADS) {
      const int64_t o = q * L_max + i;
      if (a.absorption) a.absorption[o] = NAN;
      if (a.prior_mean) a.prior_mean[o] = NAN;
      if (a.prior_sd) a.prior_sd[o] = NAN;
      if (a.fit_mean) a.fit_mean[o] = NAN;
      if (a.continuum) a.continuum[o] = NAN;
      if (a.continuum_sd) a.continuum_sd[o] = NAN;
    }
    if (a.latent) for (int c = tid; c < K; c += NTHREADS) a.latent[(int64_t)q * K + c] = NAN;
    if (tid == 0) {
      if (a.chi2) a.chi2[q] = NAN;
      if (a.log_likelihood) a.log_likelihood[q] = NAN;
      if (a.num_pixels) a.num_pixels[q] = 0;
    }
    return;
  }
  const double lo = s_lo, hi = s_hi;
  const double* wl_first = wl + first;

  // 1. absorption on the padded grid
  window_absorption(s_a, s_raw, s_mult, n_u, wl_first, lo, hi, a.pixel_spacing, a.num_lines, a.num_absorbers,
                    a.absorber_z + (int64_t)q * a.num_absorbers, a.absorber_nhi + (int64_t)q * a.num_absorbers);

  // 2. the augmented Gram [B - I | g ; . | sum r^2/d] and sum log d.  Thread tid owns entries tid + NTHREADS m of the
  // augmented upper triangle (entry NAUG: sum log d) and walks the pixels in ascending order.
  int ep[NE], eq[NE];
  double acc[NE];
#pragma unroll
  for (int m = 0; m < NE; ++m) {
    const int e = tid + NTHREADS * m;
    int p = 0;
    if (e < NAUG) {
      while (p + 1 <= K && aug_index<K>(p + 1, p + 1) <= e) ++p;
      ep[m] = p; eq[m] = p + (e - aug_index<K>(p, p));
    } else {
      ep[m] = eq[m] = -1;
    }
    acc[m] = 0.0;
  }
  for (int c0 = 0; c0 < n_u; c0 += RC_CHUNK) {
    __syncthreads();
    for (int t = tid; t < RC_CHUNK; t += NTHREADS) {
      const int i = c0 + t;
      double dinv = 0.0, logd = 0.0, r = 0.0, scale = 0.0;
      int j = 0;
      double rest = 0.0;
      bool used = false;
      if (i < n_u) {
        const double w = wl_first[i];
        rest = w / (1.0 + z_qso);
        used = !pmask[first + i] && rest >= a.min_lambda && rest <= a.max_lambda;
        if (used) {
          const PixelModel m = null_model_pixel(a.rest_wavelengths, a.mu, a.log_omega, a.n_rest, a.c_0, a.tau_0, a.beta,
                                                a.lya_wavelength, a.meanflux, w, rest, z_qso);
          const double ab = s_a[i];
          const double d = m.om2 * (ab * ab) + nv[first + i];
          r = fl[first + i] - (m.mu * m.absorb) * ab;
          dinv = 1.0 / d; logd = log(d);
          scale = m.absorb; j = m.j;
        }
      }
      s_dinv[t] = dinv; s_logd[t] = logd;
      s_u[t * KA + K] = r;
      // the K columns of a M~ for this pixel (zero when unused)
      for (int c = 0; c < K; ++c)
        s_u[t * KA + c] = used ? (interp_linear(a.rest_wavelengths, a.M + c, K, j, rest) * scale) * s_a[i] : 0.0;
    }
    __syncthreads();
    const int nc = min(RC_CHUNK, n_u - c0);
#pragma unroll
    for (int m = 0; m < NE; ++m) {
      const int p = ep[m], qq = eq[m];
      if (p >= 0) {
        double s = acc[m];
        for (int t = 0; t < nc; ++t) s = fma(s_u[t * KA + p] * s_dinv[t], s_u[t * KA + qq], s);
        acc[m] = s;
      } else if (tid + NTHREADS * m == NAUG) {
        double s = acc[m];
        for (int t = 0; t < nc; ++t) s += s_logd[t];
        acc[m] = s;
      }
    }
  }
#pragma unroll
  for (int m = 0; m < NE; ++m) {
    const int e = tid + NTHREADS * m;
    if (e <= NAUG) s_aug[e] = acc[m];
  }
  __syncthreads();

  // 3. Cholesky B = L L' (lower, left-looking: lane l owns rows j + l, j + l + 32, ...) and the two solves, in warp 0
  if (warp == 0) {
    for (int e = lane; e < K * K; e += 32) {
      const int r = e / K, c = e % K;
      if (c <= r) s_L[r * KA + c] = s_aug[aug_index<K>(c, r)] + (r == c ? 1.0 : 0.0);   // B = I + C  (:23)
    }
    __syncwarp();
    for (int j = 0; j < K; ++j) {
      double v[(K + 31) / 32];
#pragma unroll
      for (int h = 0; h < (K + 31) / 32; ++h) {
        const int r = j + lane + 32 * h;
        double s = 0.0;
        if (r < K) {
          s = s_L[r * KA + j];
          for (int m = 0; m < j; ++m) s = fma(-s_L[r * KA + m], s_L[j * KA + m], s);
        }
        v[h] = s;
      }
      const double djj = sqrt(__shfl_sync(0xffffffffu, v[0], 0));
#pragma unroll
      for (int h = 0; h < (K + 31) / 32; ++h) {
        const int r = j + lane + 32 * h;
        if (r < K) s_L[r * KA + j] = (r == j) ? djj : v[h] / djj;
      }
      if (lane == 0) s_rdiag[j] = 1.0 / djj;
      __syncwarp();
    }
    // L y = g (column sweep), then L' x = y
    for (int r = lane; r < K; r += 32) s_y[r] = s_aug[aug_index<K>(r, K)];
    __syncwarp();
    for (int j = 0; j < K; ++j) {
      const double yj = s_y[j] / s_L[j * KA + j];
      __syncwarp();
      if (lane == 0) s_y[j] = yj;
      for (int r = j + 1 + lane; r < K; r += 32) s_y[r] = fma(-s_L[r * KA + j], yj, s_y[r]);
      __syncwarp();
    }
    for (int r = lane; r < K; r += 32) s_x[r] = s_y[r];
    __syncwarp();
    for (int j = K - 1; j >= 0; --j) {
      const double xj = s_x[j] / s_L[j * KA + j];
      __syncwarp();
      if (lane == 0) s_x[j] = xj;
      for (int r = lane; r < j; r += 32) s_x[r] = fma(-s_L[j * KA + r], xj, s_x[r]);
      __syncwarp();
    }
    if (lane == 0) {
      double yy = 0.0, logdiag = 0.0;
      for (int j = 0; j < K; ++j) { yy = fma(s_y[j], s_y[j], yy); logdiag += log(s_L[j * KA + j]); }
      const double chi2 = s_aug[aug_index<K>(K, K)] - yy;                                    // :28
      const double logdet = s_aug[NAUG] + 2.0 * logdiag;                                     // :30
      if (a.chi2) a.chi2[q] = chi2;
      if (a.log_likelihood) a.log_likelihood[q] = -0.5 * (chi2 + logdet + (double)n_used * LOG_2PI);   // :32
      if (a.num_pixels) a.num_pixels[q] = n_used;
    }
    if (a.latent) for (int c = lane; c < K; c += 32) a.latent[(int64_t)q * K + c] = s_x[c];
  }
  __syncthreads();

  // 4. the per-pixel planes over the whole row
  const bool want_cond = a.fit_mean || a.continuum || a.continuum_sd || a.prior_sd;
  for (int64_t i = tid; i < L_max; i += NTHREADS) {
    double ab = NAN, pmean = NAN, psd = NAN, fmean = NAN, cont = NAN, csd = NAN;
    const int64_t iw = i - first;
    if (i < L && iw >= 0 && iw < n_u) {
      const double w = wl[i], rest = w / (1.0 + z_qso);
      if (rest >= a.min_lambda && rest <= a.max_lambda) {
        const PixelModel m = null_model_pixel(a.rest_wavelengths, a.mu, a.log_omega, a.n_rest, a.c_0, a.tau_0, a.beta,
                                              a.lya_wavelength, a.meanflux, w, rest, z_qso);
        ab = s_a[iw];
        const double mu_t = m.mu * m.absorb;
        pmean = ab * mu_t;
        if (want_cond) {
          // m_i (unsuppressed row of M): m x^, |m|^2 and z = L^-1 m by forward substitution
          double zz[K];
          double mx = 0.0, mm = 0.0, zsum = 0.0;
#pragma unroll
          for (int c = 0; c < K; ++c) {
            const double mc = interp_linear(a.rest_wavelengths, a.M + c, K, m.j, rest);
            mx = fma(mc, s_x[c], mx);
            const double mt = mc * m.absorb;
            mm = fma(mt, mt, mm);
            double s = mc;
#pragma unroll
            for (int h = 0; h < c; ++h) s = fma(-s_L[c * KA + h], zz[h], s);
            zz[c] = s * s_rdiag[c];
            zsum = fma(zz[c], zz[c], zsum);
          }
          fmean = ab * (mu_t + m.absorb * mx);
          cont = m.mu + mx;
          csd = sqrt(zsum);
          if (!pmask[i]) psd = sqrt((ab * ab) * (mm + m.om2) + nv[i]);
        }
      }
    }
    const int64_t o = q * L_max + i;
    if (a.absorption) a.absorption[o] = ab;
    if (a.prior_mean) a.prior_mean[o] = pmean;
    if (a.prior_sd) a.prior_sd[o] = psd;
    if (a.fit_mean) a.fit_mean[o] = fmean;
    if (a.continuum) a.continuum[o] = cont;
    if (a.continuum_sd) a.continuum_sd[o] = csd;
  }
}

}  // namespace gpdla
