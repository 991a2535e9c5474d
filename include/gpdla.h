/* gpdla.h -- C ABI of libgpdla.so, the B200 (sm_100a) implementation of gp_dla_detection's
 * per-quasar DLA model-selection hot path.
 *
 * Every entry point replaces one interface of the reference (paths are into the
 * jibanCat/gp_dla_detection tree):
 *
 *   gpdla_voigt / gpdla_voigt_batch_device
 *        the MEX function  profile = voigt(lambdas, z, N [, num_lines])     voigt.c:253-304
 *        (call site process_qsos.m:187-188)
 *   gpdla_set_model        load(learned_qso_model_*)  rest_wavelengths, mu, M, log_omega,
 *                          log_c_0, log_tau_0, log_beta                      process_qsos.m:29-35
 *   gpdla_set_samples      load(dla_samples)  offset_samples, log_nhi_samples, nhi_samples
 *                                                                            process_qsos.m:37-40
 *   gpdla_set_prior        prior.z_qsos, prior.dla_ind                       process_qsos.m:11-27
 *   gpdla_set_parameters   the workspace variables of set_parameters.m       set_parameters.m:5-73
 *   gpdla_process_qsos / gpdla_process_qsos_device
 *        the body of the script process_qsos.m:63-233 (per-quasar loop, sample loop calling
 *        voigt + log_mvnpdf_low_rank.m:5-34, log-sum-exp, model posteriors) plus the MAP
 *        extraction of generate_ascii_catalog.m:73-80
 *
 * Plain pointers and sizes only; no CPU fallback -- every function needs a CUDA device of
 * compute capability 10.0 and returns GPDLA_ERR_CUDA otherwise.  All functions are
 * re-entrant per context (contexts, also on different devices, may be driven from different host threads); a context
 * must not be used from two threads at once.  Every entry point leaves the caller's current CUDA device unchanged.
 */
#ifndef GPDLA_H
#define GPDLA_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GPDLA_OK 0
#define GPDLA_ERR_INVALID 1      /* bad argument (sizes, NULL, num_lines outside 1..31, num_points < 7) */
#define GPDLA_ERR_CUDA 2         /* CUDA runtime error; see gpdla_last_error */
#define GPDLA_ERR_UNSUPPORTED 3  /* configuration not compiled in (e.g. rank k) */
#define GPDLA_ERR_STATE 4        /* model / samples / prior not set */

#define GPDLA_MAX_LINES 31       /* voigt.c:16 */

typedef struct gpdla_ctx gpdla_ctx;

/* set_parameters.m:5-73 (only what the hot path reads) */
typedef struct {
  double min_lambda;            /* :33  911.75  */
  double max_lambda;            /* :34  1215.75 */
  double lya_wavelength;        /* :5   1215.6701 */
  double lyman_limit;           /* :7   911.7633 */
  double prior_z_qso_increase;  /* :56  kms_to_z(30000) */
  double min_z_cut;             /* :69  kms_to_z(3000) */
  double max_z_cut;             /* :65  kms_to_z(3000) */
  double pixel_spacing;         /* :60  1e-4 dex */
  int32_t num_lines;            /* :63  3 */
  int32_t batch_quasars;        /* quasars processed per launch group (workspace size); 0 = default */
  int32_t gram_digits;          /* arithmetic of the Gram/projection contraction (log_mvnpdf_low_rank.m:22-28):
                                 *  0 = default: exact-product INT8 tensor-core path with 6 signed 8-bit digits per
                                 *      factor (47 fractional bits; k = 20 and k = 40 -- k = 10 uses FP64 DMMA; a quasar
                                 *      with a used pixel of zero noise variance falls back to FP64 DMMA by itself)
                                 * -1 = FP64 DMMA tensor cores
                                 *  5, 6 = INT8 path with that many digits (5: 39 fractional bits, ~1e-11 relative;
                                 *      k = 40 always uses 6) */
  int32_t rest_table;           /* evaluation of the optical depth tau(lambda_obs / (1 + z_dla)) of voigt.c:282-290 inside
                                 * the fused kernels:  0 = default: per-cell polynomials of a rest-frame table wherever the
                                 *      pixel is >= 13 pixels from every line centre (5e-13 relative), direct evaluation
                                 *      of the line sum elsewhere;  -1 = direct evaluation everywhere */
} gpdla_params;

/* process_qsos.m:74-82,236-244 result variables; each array has Q entries unless noted.
 * Pointers may be NULL (that output is skipped).  Host pointers for gpdla_process_qsos,
 * device pointers for gpdla_process_qsos_device. */
typedef struct {
  double* min_z_dlas;
  double* max_z_dlas;
  double* log_priors_no_dla;
  double* log_priors_dla;
  double* log_likelihoods_no_dla;
  double* log_likelihoods_dla;
  double* log_posteriors_no_dla;
  double* log_posteriors_dla;
  double* model_posteriors;             /* [Q x 2] row-major (no DLA, DLA) */
  double* p_no_dlas;
  double* p_dlas;
  double* sample_log_likelihoods_dla;   /* [Q x S] row-major; NULL = not returned */
  double* map_z_dlas;                   /* generate_ascii_catalog.m:75-76 */
  double* map_log_nhis;                 /* generate_ascii_catalog.m:80 */
  int64_t* map_inds;                    /* 0-based arg-max sample, -1 if none */
} gpdla_results;

void gpdla_default_parameters(gpdla_params* p);

int gpdla_create(gpdla_ctx** ctx, int device);
void gpdla_destroy(gpdla_ctx* ctx);
const char* gpdla_last_error(const gpdla_ctx* ctx);
/* number of kernels this context has launched so far (for bench.py's gpu_launches) */
uint64_t gpdla_launch_count(const gpdla_ctx* ctx);

/* Optional timing of the dominant kernel (fused Voigt + Gram + Cholesky): when enabled, CUDA events
 * bracket each of its launches on the launching stream; gpdla_profile_read waits for them, returns
 * the summed milliseconds and the launch count since the last read, and resets. */
int gpdla_set_profiling(gpdla_ctx* ctx, int enable);
int gpdla_profile_read(gpdla_ctx* ctx, double* loglik_ms, int64_t* loglik_launches);

int gpdla_set_parameters(gpdla_ctx* ctx, const gpdla_params* p);
/* M is [n_rest x k], C-contiguous (MATLAB's column-major 1217 x k transposed once by the caller) */
int gpdla_set_model(gpdla_ctx* ctx, const double* rest_wavelengths, int32_t n_rest, const double* mu,
                    const double* M, int32_t k, const double* log_omega, double log_c_0, double log_tau_0,
                    double log_beta);
int gpdla_set_samples(gpdla_ctx* ctx, const double* offset_samples, const double* log_nhi_samples,
                      const double* nhi_samples, int64_t num_dla_samples);
int gpdla_set_prior(gpdla_ctx* ctx, const double* z_qsos, const uint8_t* dla_ind, int64_t n_prior);

/* Spectra are the cell arrays all_wavelengths / all_flux / all_noise_variance / all_pixel_mask of
 * preload_qsos.m:73-79 padded to [Q x L_max] row-major, with `lengths[q]` valid pixels each. */
int gpdla_process_qsos(gpdla_ctx* ctx, int64_t Q, int64_t L_max, const double* wavelengths, const double* flux,
                       const double* noise_variance, const uint8_t* pixel_mask, const int32_t* lengths,
                       const double* z_qsos, const gpdla_results* out);
/* Same with every array (inputs and outputs) already resident on the context's device;
 * `stream` is a cudaStream_t (NULL = default stream).  Asynchronous: returns after enqueueing. */
int gpdla_process_qsos_device(gpdla_ctx* ctx, int64_t Q, int64_t L_max, const double* wavelengths,
                              const double* flux, const double* noise_variance, const uint8_t* pixel_mask,
                              const int32_t* lengths, const double* z_qsos, const gpdla_results* out, void* stream);

/* ---- multi-DLA + sub-DLA + mean-flux path: multi_dlas/process_qsos_multiple_dlas_meanflux.m:100-495 ----
 *
 * gpdla_set_lls_samples   lls_nhi_samples, Z_lls, Z_dla of multi_dlas/set_lls_parameters.m:55-71
 * gpdla_process_qsos_multi(_device)
 *     the per-quasar loop ...meanflux.m:141-480 (Lyman-series mean-flux suppression :243-293, level loop
 *     :337-473 with Occam terms, z-separation filter, sub-DLA model, MAP, early exit, weighted resampling
 *     seeded by rng('default') per quasar) and the model posteriors :482-495.
 * Result variables as saved at ...meanflux.m:498-510.  Arrays with a level axis are [Q x max_dlas ...]
 * row-major; base_sample_inds and MAP_inds are 0-based (MATLAB's are 1-based).  The three large arrays may be
 * NULL (not returned).  `base_sample_inds_in` (NULL, or [Q x (max_dlas-1) x S], 0-based) replaces the
 * library's own resampling -- for bit-reproducible parity runs against another implementation. */
typedef struct {
  double* min_z_dlas;
  double* max_z_dlas;
  double* log_priors_no_dla;
  double* log_priors_lls;
  double* log_priors_dla;              /* [Q x max_dlas] */
  double* log_likelihoods_no_dla;
  double* log_likelihoods_lls;
  double* log_likelihoods_dla;         /* [Q x max_dlas] */
  double* log_posteriors_no_dla;
  double* log_posteriors_lls;
  double* log_posteriors_dla;          /* [Q x max_dlas] */
  double* model_posteriors;            /* [Q x (2 + max_dlas)]: no DLA, sub-DLA, 1..max_dlas DLAs */
  double* p_no_dlas;
  double* p_lls;
  double* p_dlas;
  double* MAP_z_dlas;                  /* [Q x max_dlas x max_dlas] */
  double* MAP_log_nhis;                /* [Q x max_dlas x max_dlas] */
  int64_t* MAP_inds;                   /* [Q x max_dlas x max_dlas], -1 = unset */
  double* sample_log_likelihoods_dla;  /* [Q x max_dlas x S]; NULL = not returned */
  double* sample_log_likelihoods_lls;  /* [Q x S]; NULL = not returned */
  int32_t* base_sample_inds;           /* [Q x (max_dlas-1) x S]; NULL = not returned */
} gpdla_multi_results;

int gpdla_set_lls_samples(gpdla_ctx* ctx, const double* lls_nhi_samples, int64_t num_dla_samples, double Z_lls,
                          double Z_dla);
int gpdla_process_qsos_multi(gpdla_ctx* ctx, int64_t Q, int64_t L_max, const double* wavelengths,
                             const double* flux, const double* noise_variance, const uint8_t* pixel_mask,
                             const int32_t* lengths, const double* z_qsos, int32_t max_dlas,
                             const int32_t* base_sample_inds_in, const gpdla_multi_results* out);
int gpdla_process_qsos_multi_device(gpdla_ctx* ctx, int64_t Q, int64_t L_max, const double* wavelengths,
                                    const double* flux, const double* noise_variance, const uint8_t* pixel_mask,
                                    const int32_t* lengths, const double* z_qsos, int32_t max_dlas,
                                    const int32_t* base_sample_inds_in, const gpdla_multi_results* out,
                                    void* stream);
/* The uniform random stream the resampling consumes (MATLAB rng('default'); rand): n values. Pure host. */
void gpdla_matlab_default_rand(double* out, int64_t n);

/* ---- spectrum preprocessing on the device (the step before the path): read_spec.m:28-38 + preload_qsos.m:26-67 ----
 * Inputs are the four columns of the SDSS speclite coadd table (read_spec.m:11-26: flux, loglam, ivar, and_mask)
 * padded to [Q x L_in] with lengths_in[q] valid pixels, and the catalogue redshifts.  Outputs are the arrays
 * all_wavelengths / all_flux / all_noise_variance / all_pixel_mask of preload_qsos.m:64-67 in the padded
 * [Q x L_out] + lengths form gpdla_process_qsos(_device) reads, all_normalizers (:49) and the updated
 * filter_flags (:36-39 bit 3 = 4: cannot normalise; :45-49 bit 4 = 8: fewer than min_num_pixels usable pixels;
 * input flags > 0 skip the quasar, :19-21).  lengths[q] = 0 for skipped quasars, -(needed) if L_out is too small.
 * Context-free; the _device entry is asynchronous on `stream` and works on the current device. */
typedef struct {
  double loading_min_lambda;         /* set_parameters.m:21  910  */
  double loading_max_lambda;         /* :22  1217 */
  double normalization_min_lambda;   /* :29  1310 */
  double normalization_max_lambda;   /* :30  1325 */
  double min_lambda;                 /* :33  911.75  */
  double max_lambda;                 /* :34  1215.75 */
  int32_t min_num_pixels;            /* :26  200 */
  int32_t reserved;
} gpdla_preload_params;
void gpdla_default_preload_parameters(gpdla_preload_params* p);
int gpdla_preload_qsos(int64_t Q, int64_t L_in, const double* flux, const double* loglam, const double* ivar,
                       const int32_t* and_mask, const int32_t* lengths_in, const double* z_qsos,
                       const uint8_t* filter_flags_in, const gpdla_preload_params* p, int64_t L_out,
                       double* wavelengths, double* out_flux, double* noise_variance, uint8_t* pixel_mask,
                       int32_t* lengths, double* normalizers, uint8_t* filter_flags);
int gpdla_preload_qsos_device(int64_t Q, int64_t L_in, const double* flux, const double* loglam, const double* ivar,
                              const int32_t* and_mask, const int32_t* lengths_in, const double* z_qsos,
                              const uint8_t* filter_flags_in, const gpdla_preload_params* p, int64_t L_out,
                              double* wavelengths, double* out_flux, double* noise_variance, uint8_t* pixel_mask,
                              int32_t* lengths, double* normalizers, uint8_t* filter_flags, void* stream);

/* ---- GP training objective on the device: objective.m:12-73 + spectrum_loss.m:14-74 ----
 * f(x) = -sum_i log N(y_i; 0, M M' + diag(sigma_i^2 + omega^2 (c_0 + 1 - exp(-tau_0 (1+z)^beta))^2)) and g = df/dx for
 *   x = [vec M (column-major num_pixels x k, as MATLAB's M(:)); log omega (num_pixels); log c_0; log tau_0; log beta]
 * (objective.m:3-6), including the Kim et al. priors on tau_0 and beta (:59-71).  The three data matrices are
 * centered_rest_fluxes, lya_1pzs, rest_noise_variances of learn_qso_model.m:36-75, [num_quasars x num_pixels]
 * row-major, NaN in centered_rest_fluxes = pixel not observed (objective.m:42).  g has the layout of x.
 * Context-free; the _device entry (device pointers for data, x, f, g) is asynchronous on `stream`.  A spectrum's pixel
 * arrays live in shared memory (about 20 bytes per pixel): a num_pixels beyond the device's opt-in limit (near 9 700 at
 * k = 40 on 227 KB) returns GPDLA_ERR_INVALID before anything is allocated or launched. */
/* The Lyman-series variant the multi-DLA model is trained with: multi_dlas/objective_lyseries.m:13-87 +
 * multi_dlas/spectrum_loss_lyseries.m:14-91.  Same x, data matrices and outputs; the effective optical depth sums the
 * first num_forest_lines series members (all_transition_wavelengths, all_oscillator_strengths of
 * set_parameters_multi.m:76-142, host arrays) that lie below the quasar, whose 1 + z is the LAST column of its lya_1pzs
 * row (objective_lyseries.m:46).  num_forest_lines = 0 is gpdla_objective. */
int gpdla_objective_lyseries(int64_t num_quasars, int32_t num_pixels, int32_t k, const double* centered_rest_fluxes,
                             const double* lya_1pzs, const double* rest_noise_variances, int32_t num_forest_lines,
                             const double* all_transition_wavelengths, const double* all_oscillator_strengths,
                             const double* x, double* f, double* g);
int gpdla_objective_lyseries_device(int64_t num_quasars, int32_t num_pixels, int32_t k, const double* centered_rest_fluxes,
                                    const double* lya_1pzs, const double* rest_noise_variances, int32_t num_forest_lines,
                                    const double* all_transition_wavelengths, const double* all_oscillator_strengths,
                                    const double* x, double* f, double* g, void* stream);
int gpdla_objective(int64_t num_quasars, int32_t num_pixels, int32_t k, const double* centered_rest_fluxes,
                    const double* lya_1pzs, const double* rest_noise_variances, const double* x, double* f, double* g);
int gpdla_objective_device(int64_t num_quasars, int32_t num_pixels, int32_t k, const double* centered_rest_fluxes,
                           const double* lya_1pzs, const double* rest_noise_variances, const double* x, double* f,
                           double* g, void* stream);

/* ---- GP training set on the device: learn_qso_model.m:36-75 (+ the nanstd of :82-95) ----
 * Inputs are the training spectra in the padded [N x L_max] form of gpdla_process_qsos (observed wavelengths, flux,
 * noise variance, pixel mask, lengths, z_qsos) and the model grid rest_wavelengths [num_pixels] (strictly increasing).
 * Per spectrum: emitted wavelengths lambda / (1 + z); flux and noise variance NaN where masked; each of
 * 1 + (lambda - lya_wavelength) / lya_wavelength, flux and noise variance linearly interpolated (interp1) onto the grid,
 * NaN outside the spectrum or next to a NaN; every grid point whose interpolated noise variance exceeds
 * max_noise_variance set to NaN in all three outputs (:66-69).  Outputs: lya_1pzs, centered_rest_fluxes (rest fluxes
 * minus mu), rest_noise_variances, [N x num_pixels] row-major; per rest pixel mu = nanmean of the rest fluxes,
 * num_observed = their non-NaN count, std_dev = nanstd (n - 1) of the centred fluxes.  A spectrum with lengths < 2 gives
 * an all-NaN row.  The host entry checks lengths in [0, L_max] and the grid, and returns GPDLA_ERR_INVALID (outputs
 * written) if a rest pixel is observed fewer than 2 times.  Context-free; the _device entry is asynchronous on `stream`
 * and works on the current device. */
int gpdla_training_set(int64_t N, int64_t L_max, const double* wavelengths, const double* flux,
                       const double* noise_variance, const uint8_t* pixel_mask, const int32_t* lengths,
                       const double* z_qsos, const double* rest_wavelengths, int32_t num_pixels,
                       double lya_wavelength, double max_noise_variance,
                       double* lya_1pzs, double* centered_rest_fluxes, double* rest_noise_variances,
                       double* mu, double* std_dev, int32_t* num_observed);
int gpdla_training_set_device(int64_t N, int64_t L_max, const double* wavelengths, const double* flux,
                              const double* noise_variance, const uint8_t* pixel_mask, const int32_t* lengths,
                              const double* z_qsos, const double* rest_wavelengths, int32_t num_pixels,
                              double lya_wavelength, double max_noise_variance,
                              double* lya_1pzs, double* centered_rest_fluxes, double* rest_noise_variances,
                              double* mu, double* std_dev, int32_t* num_observed, void* stream);
/* The covariance pca(X, 'rows', 'pairwise') decomposes (learn_qso_model.m:82-95): X [N x P] row-major, NaN = not
 * observed; X~ = X - nanmean(X) column-wise; cov[p, q] = sum over the rows observed in both columns of X~_rp X~_rq,
 * divided by (counts[p, q] - 1), NaN where counts < 2.  cov, counts: [P x P] row-major, symmetric.  FP64 tensor cores;
 * every sum has a fixed order, so repeated calls return the same bits.  Context-free; the _device entry is asynchronous on
 * `stream`. */
int gpdla_pairwise_covariance(int64_t N, int32_t P, const double* X, double* cov, int32_t* counts);
int gpdla_pairwise_covariance_device(int64_t N, int32_t P, const double* X, double* cov, int32_t* counts, void* stream);

/* ---- Training set of the multi-DLA (mean-flux) null model: multi_dlas/learn_qso_model_meanflux.m ----
 * The gpdla_training_set arguments (max_noise_variance is 3^2 for this model, set_parameters_multi.m:37) plus
 * num_forest_lines (0..31; 31 in the reference) and the nullable output lya_absorption [N x num_pixels].  After the
 * interpolation and the noisy-pixel rule (applied to the noise variance before the correction), each of the first
 * num_forest_lines Lyman-series members l gives 1 + z_l = interp1(x, 1 + (lambda - lambda_l) / lambda_l, r) with the same
 * interval and weight; total = sum_l kim_tau_l (1 + z_l)^3.65 in ascending l, kim_tau_l = 0.0023 f_l / f_lya * lambda_l /
 * lya_wavelength (the table the multi-DLA inference uses); the Lya term always counts, a term l >= 1 only where
 * 1 + z_l <= 1 + z_qso; NaN terms are skipped, so lya_absorption = exp(-total) is 1 where nothing is observed.  Rest
 * fluxes are divided by lya_absorption and rest noise variances by lya_absorption^2 before mu, the centring and std_dev;
 * lya_1pzs is not corrected.  num_forest_lines = 0 gives the bits of gpdla_training_set.  Checks, errors and the
 * GPDLA_ERR_INVALID of a rest pixel observed fewer than 2 times as gpdla_training_set. */
int gpdla_training_set_lyseries(int64_t N, int64_t L_max, const double* wavelengths, const double* flux,
                                const double* noise_variance, const uint8_t* pixel_mask, const int32_t* lengths,
                                const double* z_qsos, const double* rest_wavelengths, int32_t num_pixels,
                                double lya_wavelength, double max_noise_variance, int32_t num_forest_lines,
                                double* lya_1pzs, double* centered_rest_fluxes, double* rest_noise_variances,
                                double* lya_absorption, double* mu, double* std_dev, int32_t* num_observed);
int gpdla_training_set_lyseries_device(int64_t N, int64_t L_max, const double* wavelengths, const double* flux,
                                       const double* noise_variance, const uint8_t* pixel_mask, const int32_t* lengths,
                                       const double* z_qsos, const double* rest_wavelengths, int32_t num_pixels,
                                       double lya_wavelength, double max_noise_variance, int32_t num_forest_lines,
                                       double* lya_1pzs, double* centered_rest_fluxes, double* rest_noise_variances,
                                       double* lya_absorption, double* mu, double* std_dev, int32_t* num_observed,
                                       void* stream);
/* The matrix learn_qso_model_meanflux.m hands to pca(..., 'rows', 'complete'): out = X with each row's NaNs replaced by
 * that row's nanmedian (MATLAB's median: for an even count meanof(a, b) = a + (b - a) / 2, or (a + b) / 2 when
 * sign(a) ~= sign(b) or either is infinite).  An all-NaN row stays NaN, so every row of out is complete or all NaN and
 * gpdla_pairwise_covariance of out is the covariance of its complete rows.  X, out: [N x P] row-major, 1 <= P <= 16384;
 * out may alias X.  Deterministic (no atomics).  Context-free; the _device entry is asynchronous on `stream`. */
int gpdla_row_nanmedian_fill(int64_t N, int32_t P, const double* X, double* out);
int gpdla_row_nanmedian_fill_device(int64_t N, int32_t P, const double* X, double* out, void* stream);

/* Population statistics of the single-DLA catalogue (the additive sums behind CDDF_analysis/calc_cddf.py: column density
 * distribution, dN/dX, Omega_DLA; Bird, Garnett & Ho 2017) from one gpdla_process_qsos call's outputs with the same
 * samples: sample_log_likelihoods_dla [Q x S], p_dlas, min_z_dlas, max_z_dlas [Q], the nullable uint8 mask `select`
 * [Q], and offset_samples, log_nhi_samples, nhi_samples [S].  Quasar i contributes iff select[i] (default 1),
 * isfinite(p_dlas[i]), max_z > min_z and its row's log-sum-exp is finite; w_ij is its normalised sample posterior,
 * z_ij = min_z + (max_z - min_z) offset_j rounded as map_z_dlas, bins are half-open [lo, hi).  `sums` (in/out, float64,
 * 2 n_z n_nhi + 5 n_z + 1 entries) is ADDED to, in this layout:
 *   counts[n_z][n_nhi] = sum q, counts_var[n_z][n_nhi] = sum q(1-q), q = p sum_j w_j [z_j in b, log N_j in c]
 *   dla[n_z] = sum d, dla_var[n_z] = sum d(1-d), d = p sum_j w_j [z_j in b, log N_j >= dla_log_nhi_min]
 *   nhi[n_z] = sum e, nhi_var[n_z] = sum (e2 - e^2), e = p sum_j w_j N_j [...], e2 = p sum_j w_j N_j^2 [...]
 *   path[n_z] = sum dX, flat LambdaCDM X(z) = 2 / (3 omega_m) sqrt(omega_m (1+z)^3 + 1 - omega_m), clipped to
 *               [min_z, max_z] of each quasar;   num_quasars.
 * Sums of disjoint sets of quasars add; variances add across quasars, never across z bins (one quasar's cells are
 * exclusive), so an all-z statistic needs one z bin.  z_edges [n_z + 1], log_nhi_edges [n_nhi + 1]: host arrays,
 * finite and strictly increasing; 1 <= n_z <= 64, 1 <= n_nhi <= 128, omega_m in (0, 1], else GPDLA_ERR_INVALID before
 * any CUDA call.  No atomics: repeated calls give the same bits.  Context-free, on the current device; the _device entry
 * takes device arrays and is asynchronous on `stream`, the other entry host arrays. */
int gpdla_dla_statistics(int64_t Q, int64_t S, const double* sample_log_likelihoods_dla, const double* p_dlas,
                         const double* min_z_dlas, const double* max_z_dlas, const uint8_t* select,
                         const double* offset_samples, const double* log_nhi_samples, const double* nhi_samples,
                         int32_t n_z, const double* z_edges, int32_t n_nhi, const double* log_nhi_edges,
                         double dla_log_nhi_min, double omega_m, double* sums);
int gpdla_dla_statistics_device(int64_t Q, int64_t S, const double* sample_log_likelihoods_dla, const double* p_dlas,
                                const double* min_z_dlas, const double* max_z_dlas, const uint8_t* select,
                                const double* offset_samples, const double* log_nhi_samples, const double* nhi_samples,
                                int32_t n_z, const double* z_edges, int32_t n_nhi, const double* log_nhi_edges,
                                double dla_log_nhi_min, double omega_m, double* sums, void* stream);

/* Population statistics of the multi-DLA catalogue (Ho et al. 2021) from one gpdla_process_qsos_multi(_device) call's
 * outputs with the same samples: sample_log_likelihoods_dla [Q x max_dlas x S], base_sample_inds
 * [Q x (max_dlas-1) x S] (0-based; NULL only when max_dlas == 1), model_posteriors [Q x (2 + max_dlas)] (no DLA,
 * sub-DLA, 1..max_dlas DLAs), min_z_dlas, max_z_dlas [Q], the nullable uint8 mask `select` [Q], and offset_samples,
 * log_nhi_samples, nhi_samples [S].  Per quasar the model is a mixture: model M with probability p_M; under j DLAs,
 * sample i with its normalised weight w_ji (NaN entries, the z-separation filter's, weigh 0), which places j absorbers
 * at samples i, base_sample_inds[0][i], ..., base_sample_inds[j-2][i].  The no-DLA and sub-DLA models place none.
 * Quasar q contributes iff select[q] (default 1), every entry of its model_posteriors row is finite, max_z > min_z,
 * and every level with p_j > 0 has a finite maximum log-likelihood and partner indices in [0, S); levels with p_j == 0
 * are skipped.  `sums` (in/out, float64, the layout of gpdla_dla_statistics) is ADDED to, with the exact mixture mean
 * and variance of each per-quasar count:
 *   counts / counts_var[n_z][n_nhi]   E[X], E[X^2] - E[X]^2 of X = the number of absorbers in the (z, log N) cell
 *   dla / dla_var[n_z]                the same of D = the number of absorbers in the z bin with log N >= dla_log_nhi_min
 *   nhi / nhi_var[n_z]                the same of E = the sum of N_HI over those absorbers
 *   path[n_z], num_quasars            as gpdla_dla_statistics.
 * With max_dlas == 1 this is the single-DLA statistic.  Every argument check of gpdla_dla_statistics applies, and
 * 1 <= max_dlas <= 4; else GPDLA_ERR_INVALID before any CUDA call.  The host entry also rejects a base_sample_inds
 * entry outside [0, S).  No atomics: repeated calls give the same bits, and the host entry those of the _device entry.
 * Context-free, on the current device; the _device entry takes device arrays and is asynchronous on `stream`. */
int gpdla_multi_dla_statistics(int64_t Q, int64_t S, int32_t max_dlas, const double* sample_log_likelihoods_dla,
                               const int32_t* base_sample_inds, const double* model_posteriors,
                               const double* min_z_dlas, const double* max_z_dlas, const uint8_t* select,
                               const double* offset_samples, const double* log_nhi_samples, const double* nhi_samples,
                               int32_t n_z, const double* z_edges, int32_t n_nhi, const double* log_nhi_edges,
                               double dla_log_nhi_min, double omega_m, double* sums);
int gpdla_multi_dla_statistics_device(int64_t Q, int64_t S, int32_t max_dlas, const double* sample_log_likelihoods_dla,
                                      const int32_t* base_sample_inds, const double* model_posteriors,
                                      const double* min_z_dlas, const double* max_z_dlas, const uint8_t* select,
                                      const double* offset_samples, const double* log_nhi_samples,
                                      const double* nhi_samples, int32_t n_z, const double* z_edges, int32_t n_nhi,
                                      const double* log_nhi_edges, double dla_log_nhi_min, double omega_m,
                                      double* sums, void* stream);

/* ---- Per-quasar summaries of the absorber posterior: error bars, effective sample size and the DLA-threshold mass
 * that the point estimates (map_z_dlas, map_log_nhis, MAP_*) do not carry ----
 * Single-DLA model.  Inputs as gpdla_dla_statistics takes them: sample_log_likelihoods_dla [Q x S] (gpdla_process_qsos
 * output), min_z_dlas, max_z_dlas [Q], offset_samples, log_nhi_samples [S].  The sample posterior of quasar q is
 * w_i = exp(ll_i - max ll) (NaN and -inf entries weigh 0); the samples are prior draws, so this is the DLA-model
 * posterior over the sample set (process_qsos.m:203-210).  z_i = min_z + (max_z - min_z) * offset_i, each operation
 * rounded, as map_z_dlas.  out [Q x (7 + 2 num_quantiles)], float64, per quasar:
 *   ess                    Kish's effective sample size (sum w)^2 / sum w^2
 *   z_mean, z_sd           posterior mean and standard deviation of z_DLA (two-pass central moments)
 *   log_nhi_mean, log_nhi_sd, z_log_nhi_cov   the same of log10 N_HI, and the covariance of the two
 *   mass_above_threshold   sum over log N_i >= log_nhi_threshold of w_i / sum w (p_dla times it: a DLA proper)
 *   z_quantiles[P], log_nhi_quantiles[P]   the lower inverse CDF at quantiles[p]: the value of the first sample, in
 *                          value order, whose cumulative weight reaches quantiles[p] * (the scan's total weight)
 * A quasar with no finite weight, or with max_z_dlas <= min_z_dlas (or NaN), gets a NaN record.  Checks before any
 * CUDA call, else GPDLA_ERR_INVALID: 0 <= Q < 2^31, 1 <= S < 2^31, 1 <= num_quantiles <= 16, every quantile inside
 * (0, 1) (NaN is not), a finite log_nhi_threshold, no NULL array (the per-quasar ones may be NULL when Q == 0).
 * No atomics: repeated calls give the same bits, and the host entry those of the _device entry, which takes device
 * arrays (quantiles stays a host array) and is asynchronous on `stream`.  Context-free, on the current device. */
int gpdla_dla_posteriors(int64_t Q, int64_t S, const double* sample_log_likelihoods_dla, const double* min_z_dlas,
                         const double* max_z_dlas, const double* offset_samples, const double* log_nhi_samples,
                         int32_t num_quantiles, const double* quantiles, double log_nhi_threshold, double* out);
int gpdla_dla_posteriors_device(int64_t Q, int64_t S, const double* sample_log_likelihoods_dla,
                                const double* min_z_dlas, const double* max_z_dlas, const double* offset_samples,
                                const double* log_nhi_samples, int32_t num_quantiles, const double* quantiles,
                                double log_nhi_threshold, double* out, void* stream);
/* Multi-DLA model (Ho et al. 2021).  sample_log_likelihoods_dla [Q x max_dlas x S] and base_sample_inds
 * [Q x (max_dlas - 1) x S] (0-based; may be NULL when max_dlas == 1) in the layout of gpdla_process_qsos_multi: sample
 * i of level j places j absorbers, at samples i and base_sample_inds[0..j-2][i].  Per level j = 1..max_dlas, with
 * w_ji = exp(ll_ji - max_i ll_ji): ess_j, and for the absorber of rank r < j in ascending z (ties broken by log N, then
 * slot) the posterior mean and standard deviation of its z and log N (slots are exchangeable under the resampling,
 * ranks are not).  out [Q x (J + 4 J (J + 1) / 2)], level-major: level j holds ess_j, then (z_mean, z_sd,
 * log_nhi_mean, log_nhi_sd) of ranks 0..j-1 (44 doubles at J = 4).  A level with no finite weight, or whose partner
 * rows hold an index outside [0, S), is NaN, the other levels are not; max_z_dlas <= min_z_dlas makes the record NaN.
 * Quantiles of the ranks and their DLA-threshold mass are gpdla_multi_dla_posterior_quantiles' record.  Checks as
 * above plus 1 <= max_dlas <= 4; partner indices are not rejected (they make a level NaN).  No atomics; the host entry
 * gives the bits of the _device entry, which is asynchronous on `stream`. */
int gpdla_multi_dla_posteriors(int64_t Q, int64_t S, int32_t max_dlas, const double* sample_log_likelihoods_dla,
                               const int32_t* base_sample_inds, const double* min_z_dlas, const double* max_z_dlas,
                               const double* offset_samples, const double* log_nhi_samples, double* out);
int gpdla_multi_dla_posteriors_device(int64_t Q, int64_t S, int32_t max_dlas, const double* sample_log_likelihoods_dla,
                                      const int32_t* base_sample_inds, const double* min_z_dlas,
                                      const double* max_z_dlas, const double* offset_samples,
                                      const double* log_nhi_samples, double* out, void* stream);
/* Credible intervals of every absorber of the multi-DLA model.  Arguments as gpdla_multi_dla_posteriors, plus
 * num_quantiles, quantiles and log_nhi_threshold as gpdla_dla_posteriors.  Per level j = 1..max_dlas and rank r < j
 * (the absorber of rank r in ascending z, ties by log N, then slot, as above), under w_ji = exp(ll_ji - max_i ll_ji):
 *   mass_above_threshold   sum of w_ji over the samples whose rank-r absorber has log N >= log_nhi_threshold, / sum w
 *   z_quantiles[P], log_nhi_quantiles[P]   the lower inverse CDF of the rank-r absorber's z and log N: the value at the
 *                          first position, in value order, whose cumulative fixed-point weight reaches quantiles[p]
 *                          times the scan's total
 * out [Q x J (J + 1) / 2 x (1 + 2 num_quantiles)], level-major, then rank (110 doubles at J = 4, P = 5).  Every
 * absorber is one of the samples, so its value order is the samples' order by offset (z) or by log N for every quasar,
 * and the CDF is a histogram over the S sample positions.  Its bins hold sum floor(w 2^F) exactly, as uint64, with
 * F = 63 - ceil(log2 S) (49 at S = 10^4, 46 at S = 10^5); the largest weight is 1, so each cumulative fraction is within
 * S 2^-F of that of the float weights (1.8e-11 at S = 10^4, 1.4e-9 at S = 10^5): a reported quantile is a value whose
 * cumulative float weight lies within S 2^-F + 1e-12 of quantiles[p] times the total.  The mass is a float sum, as in
 * gpdla_dla_posteriors.  NaN as gpdla_multi_dla_posteriors: a level with no finite weight or a partner row outside
 * [0, S) is NaN, the other levels keep their bits; max_z_dlas <= min_z_dlas makes the record NaN.  Checks before any
 * CUDA call: those of both entries above.  Integer atomics only: repeated calls give the same bits, and the host
 * entry those of the _device entry, which is asynchronous on `stream` (quantiles stays a host array). */
int gpdla_multi_dla_posterior_quantiles(int64_t Q, int64_t S, int32_t max_dlas, const double* sample_log_likelihoods_dla,
                                        const int32_t* base_sample_inds, const double* min_z_dlas,
                                        const double* max_z_dlas, const double* offset_samples,
                                        const double* log_nhi_samples, int32_t num_quantiles, const double* quantiles,
                                        double log_nhi_threshold, double* out);
int gpdla_multi_dla_posterior_quantiles_device(int64_t Q, int64_t S, int32_t max_dlas,
                                               const double* sample_log_likelihoods_dla,
                                               const int32_t* base_sample_inds, const double* min_z_dlas,
                                               const double* max_z_dlas, const double* offset_samples,
                                               const double* log_nhi_samples, int32_t num_quantiles,
                                               const double* quantiles, double log_nhi_threshold, double* out,
                                               void* stream);

/* ---- The fitted model of each quasar under chosen absorbers: what CDDF_analysis/qso_loader.py:1654-1774
 * (plot_this_mu) draws, on the device, with the hot path's own model evaluation ----
 * Spectra as gpdla_process_qsos takes them.  absorber_z, absorber_nhi: [Q x num_absorbers] (N in cm^-2, as voigt and
 * nhi_samples take it); an entry with NaN z is no absorber, so rows may hold fewer; 0 <= num_absorbers <= 4, and the two
 * arrays may be NULL only when it is 0.  meanflux = 1 evaluates the null model of the multi-DLA path (Lyman-series
 * mean-flux suppression s and noise scaling), 0 that of process_qsos.m (s = 1).  For quasar q, over the pixels of the
 * modelled window (min_lambda <= lambda / (1 + z_qso) <= max_lambda, masked ones included):
 *   mu~, M~, om2~   the interpolated model exactly as the hot path evaluates it, suppressed by s
 *   a               the product of the absorbers' instrument-convolved profiles on the padded window grid (voigt.c,
 *                   params.num_lines lines, optical depth always evaluated directly)
 * and over the used pixels (window, not masked), d = a^2 om2~ + v, r = y - a mu~, B = I + (a M~)' D^-1 (a M~),
 * g = (a M~)' D^-1 r.  Outputs, each nullable (skipped when NULL); planes are [Q x L_max], NaN outside the window and
 * past lengths[q]:
 *   absorption      a
 *   prior_mean      a mu~
 *   prior_sd        sqrt(a^2 (sum_c M~_c^2 + om2~) + v); NaN on masked pixels
 *   fit_mean        a (mu~ + M~ x^), the conditional mean of the smooth part
 *   continuum       mu + M x^: the emitted continuum, without the forest's mean absorption and the absorbers
 *   continuum_sd    sqrt(m' B^-1 m), m the unsuppressed interpolated row of M
 *   latent [Q x k]  x^ = B^-1 g
 *   chi2 [Q]        sum r^2/d - g' B^-1 g
 *   log_likelihood  -1/2 (chi2 + sum log d + 2 sum log L_ii + n log 2pi), B = L L': the hot path's Gaussian log-density
 *   num_pixels      n (int32)
 * A quasar without a used pixel gets NaN everywhere and num_pixels = 0.  Needs a model (GPDLA_ERR_STATE without one);
 * samples and prior are not read.  k = 10, 20, 40 (else GPDLA_ERR_UNSUPPORTED); L_max is bounded by one CTA's shared
 * memory (about 20 000 pixels).  The argument checks (and, in the host entry, that every finite z is > -1 with a finite
 * N >= 0) come before any CUDA call.  No atomics: repeated calls give the same bits, and the host entry those of the
 * _device entry, which takes device arrays and is asynchronous on `stream`. */
typedef struct {
  double* absorption;
  double* prior_mean;
  double* prior_sd;
  double* fit_mean;
  double* continuum;
  double* continuum_sd;
  double* latent;
  double* chi2;
  double* log_likelihood;
  int32_t* num_pixels;
} gpdla_reconstruction;
int gpdla_reconstruct(gpdla_ctx* ctx, int64_t Q, int64_t L_max, const double* wavelengths, const double* flux,
                      const double* noise_variance, const uint8_t* pixel_mask, const int32_t* lengths,
                      const double* z_qsos, int32_t meanflux, int32_t num_absorbers, const double* absorber_z,
                      const double* absorber_nhi, const gpdla_reconstruction* out);
int gpdla_reconstruct_device(gpdla_ctx* ctx, int64_t Q, int64_t L_max, const double* wavelengths, const double* flux,
                             const double* noise_variance, const uint8_t* pixel_mask, const int32_t* lengths,
                             const double* z_qsos, int32_t meanflux, int32_t num_absorbers, const double* absorber_z,
                             const double* absorber_nhi, const gpdla_reconstruction* out, void* stream);

/* ---- Draws from the learned model: mock spectra from the prior predictive, or absorbers injected into spectra,
 * with the truth of every draw ----
 * Spectra as gpdla_process_qsos takes them (flux_in is read only when injecting).  For quasar q, over the pixels of the
 * modelled window (min_lambda <= lambda / (1 + z_qso) <= max_lambda, masked ones included), mu~, M~ and om2~ are the
 * null model exactly as gpdla_reconstruct evaluates it (model 0: that of process_qsos.m, s = 1; model 1: the mean-flux
 * null model of the multi-DLA path), and a is the product of the absorbers' instrument-convolved profiles on the
 * padded window grid (params.num_lines lines, optical depth evaluated directly), bit-equal to gpdla_reconstruct's
 * absorption plane for the same absorbers.  Modes:
 *   draw    y = a (mu~ + M~ xi + om2~^(1/2) e1) + v^(1/2) e2,  xi ~ N(0, I_k) per quasar, e1, e2 ~ N(0, 1) per pixel:
 *           an exact draw from the Gaussian whose density the hot path evaluates (log_mvnpdf_low_rank.m).  Pixels
 *           outside the window are NaN (the model does not define them), pixels past lengths[q] are 0.
 *   inject  y' = a y + ((1 - a^2) v)^(1/2) e2 on the caller's flux y (the noise variance stays v; where a^2 >= 1 the
 *           noise term is 0): if y is a draw from the model, y' is one with the absorbers added.  Pixels outside the
 *           window and past lengths[q] are copied.
 * Absorbers are either given (from_prior = 0: absorber_z, absorber_nhi [Q x num_absorbers], 0 <= num_absorbers <= 4,
 * NaN z = none; the conventions and checks of gpdla_reconstruct), or drawn from the model's own prior (from_prior = 1),
 * discretised on the loaded samples exactly as the evidence integrates over them, with min_z, max_z the used-pixel
 * range of processing (set_parameters.m:65-73) and z_i = min_z + (max_z - min_z) offset_i rounded as map_z_dlas:
 *   model 0   one DLA with probability exp(log_prior_dla) (process_qsos.m:122-131, from the prior catalogue), at a
 *             uniformly drawn sample i: (z_i, nhi_samples[i]).  Its z is bit-equal to the z processing gives sample i.
 *   model 1   no DLA, sub-DLA or j = 1..max_dlas DLAs with the priors of ...meanflux.m:190-216.  A sub-DLA is a
 *             uniform sample i at (z_i, lls_nhi_samples[i]); j DLAs are j i.i.d. uniform samples, the whole set
 *             redrawn (up to 64 attempts) until every z gap is >= kms_to_z(3000), the separation filter of the level
 *             evidence; after 64 failures the quasar is flagged (truth_model = -2), never silently changed.  The
 *             multi-DLA evidence is an importance-sampled estimate (resampled partners, Occam terms), so its posterior
 *             calibration against these draws is close to, not exactly, an identity.
 * A quasar without a used pixel gets a NaN flux and absorption row (in both modes and with both sources); with the
 * prior source so does one whose model probabilities are not finite (no prior quasar below its z), truth_model = -1.
 * Truth (prior source only; TW = max_dlas for model 1, 1 for model 0):
 *   truth_model [Q] int32      -2 no separated set, -1 no draw, 0 no absorber, 1 sub-DLA, 1 + j: j DLAs
 *   truth_inds [Q x TW] int64  0-based sample indices in the caller's sample order, -1 for an empty slot
 *   truth_z, truth_log_nhi [Q x TW]  NaN for an empty slot; log_nhi_samples[i] for a DLA, log10(lls_nhi_samples[i]) for
 *                              a sub-DLA (the context holds no log copy of the sub-DLA samples)
 * Absorbers are listed in ascending z (ties in slot order), the rank order of the multi-DLA posterior entries.
 * Random numbers: Philox4x32-10 (10 rounds, multipliers 0xD2511F53 / 0xCD9E8D57, Weyl constants 0x9E3779B9 /
 * 0xBB67AE85; the bits of curand_Philox4x32_10), key = seed (low word first), counter = (element, stream, g_lo, g_hi)
 * with g = first_quasar + q, the quasar's index in the whole catalogue.  A draw therefore depends on (seed, g, stream,
 * element) only -- not on the batch split, grid or GPU count: shards with their first_quasar draw the bits of the
 * whole.  The output words r.x..r.w make W0 = r.y:r.x and W1 = r.w:r.z (64 bits each).  Layout:
 *   stream 0, element 0                   the model choice u = ((W0 >> 11) + 0.5) 2^-53: the first model m with
 *                                         u < sum_{<= m} p, else the last
 *   stream 1, element 4 attempt + slot    a sample index __umul64hi(W0, S)
 *   stream 2, element c                   latent xi_2c, xi_2c+1
 *   stream 3, element i (pixel in row)    e1, e2
 * Normals are Box-Muller on the uniforms of W0 and W1: r = sqrt(-2 log u0), r cospi(2 u1), r sinpi(2 u1).  This layout
 * changes only together with the test oracle (oracle/draw_spectra_oracle.py).
 * Options: model 0 or 1; max_dlas 1..4 (model 1); inject 0/1; from_prior 0/1; first_quasar >= 0.  Outputs: flux
 * [Q x L_max] (required), absorption [Q x L_max] (nullable, NaN outside the window and past lengths[q]) and, with
 * from_prior, the four truth arrays (required).  GPDLA_ERR_STATE without a model, and with from_prior also without
 * samples and prior, and for model 1 without the sub-DLA samples.  GPDLA_ERR_INVALID: flux_in NULL when injecting,
 * given absorbers with from_prior, first_quasar < 0, a truth pointer NULL with from_prior, and the checks of
 * gpdla_reconstruct; all before any CUDA call.  k = 10, 20, 40 (else GPDLA_ERR_UNSUPPORTED), L_max bounded by one
 * CTA's shared memory (about 20 000 pixels).  No atomics: repeated calls give the same bits, and the host entry those
 * of the _device entry, which takes device arrays and is asynchronous on `stream`. */
typedef struct {
  uint64_t seed;
  int64_t first_quasar;
  int32_t model;
  int32_t max_dlas;
  int32_t inject;
  int32_t from_prior;
  int32_t num_absorbers;
  int32_t reserved;
  const double* absorber_z;
  const double* absorber_nhi;
} gpdla_draw_options;
typedef struct {
  double* flux;
  double* absorption;
  int32_t* truth_model;
  int64_t* truth_inds;
  double* truth_z;
  double* truth_log_nhi;
} gpdla_draw_outputs;
int gpdla_draw_spectra(gpdla_ctx* ctx, int64_t Q, int64_t L_max, const double* wavelengths, const double* flux_in,
                       const double* noise_variance, const uint8_t* pixel_mask, const int32_t* lengths,
                       const double* z_qsos, const gpdla_draw_options* options, const gpdla_draw_outputs* out);
int gpdla_draw_spectra_device(gpdla_ctx* ctx, int64_t Q, int64_t L_max, const double* wavelengths,
                              const double* flux_in, const double* noise_variance, const uint8_t* pixel_mask,
                              const int32_t* lengths, const double* z_qsos, const gpdla_draw_options* options,
                              const gpdla_draw_outputs* out, void* stream);

/* voigt.c:253-304: profile has num_points - 6 entries.  Host buffers; runs on the current device. */
int gpdla_voigt(const double* lambdas, int64_t num_points, double z, double N, int32_t num_lines, double* profile);
/* Batched, device buffers: profile[s, :] = voigt(lambdas, z[s], N[s], num_lines), [S x (num_points-6)] */
int gpdla_voigt_batch_device(const double* lambdas, int64_t num_points, const double* z, const double* N,
                             int64_t S, int32_t num_lines, double* profile, void* stream);

/* The rest-frame table of tau / N the fused kernels use (see gpdla_params.rest_table), as the library builds it for
 * `num_lines` lines and cells of `pixel_spacing` dex, for verification: cell c is centred at rest wavelength
 * lambda_lo * exp(c * h) and holds the coefficients coef[p * ncell + c], p = 0..degree, of a polynomial in
 * s = ln(lambda / centre) / h, |s| <= 1/2; NaN marks the cells left to direct evaluation.  `coef` may be NULL
 * (sizes only); otherwise it must hold (degree + 1) * ncell doubles (call once with NULL to size it).  Pure host. */
int gpdla_rest_table(int32_t num_lines, double pixel_spacing, double* coef, int32_t* ncell, int32_t* degree,
                     double* h, double* lambda_lo);

/* Page-locked host memory for the buffers of gpdla_process_qsos (optional: pageable buffers work, pinned ones let
 * the result copies overlap the next batch).  cudaHostAlloc / cudaFreeHost behind a C signature. */
int gpdla_host_alloc(void** ptr, uint64_t bytes);
void gpdla_host_free(void* ptr);

/* Lyman-series constants as the library computes them (voigt.c:31-220,242-251), for verification:
 * each output has GPDLA_MAX_LINES entries (instrument_profile: 7).  Pure host function. */
void gpdla_line_constants(double* transition_wavelengths, double* leading_constants, double* gammas,
                          double* instrument_profile);

#ifdef __cplusplus
}
#endif
#endif /* GPDLA_H */
