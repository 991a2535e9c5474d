r"""TEST INFRASTRUCTURE (oracle): literal NumPy restatement of the training set and PCA initialisation of the
multi-DLA (mean-flux) null model, one spectrum at a time, in the operation order the CUDA kernels follow.

multi_dlas/learn_qso_model_meanflux.m builds the multi-DLA model's training set as learn_qso_model.m does
(``training_set_oracle``, steps 1-7 there) except for four steps:

1'. step 1 as in training_set_oracle, and for each of the first num_forest_lines (31) Lyman-series members l
   (set_parameters_multi.m:77-109, Angstrom) 1 + z_l = interp1(x, 1 + (lambda - lambda_l) / lambda_l, r) with the same j and t;
2'. noisy pixels with max_noise_variance = 3^2 (set_parameters_multi.m:37); NaN in every 1 + z_l as well;
3'. mean-flux correction (Kim et al. 2007, fixed prev_tau_0 = 0.0023, prev_beta = 3.65): total = nansum over l, in
   ascending l, of kim_tau_l (1 + z_l)^prev_beta with kim_tau_l = prev_tau_0 f_l / f_lya * lambda_l / lya_wavelength; a
   term l >= 1 counts only where 1 + z_l <= 1 + z_qso; lya_absorption = exp(-total); rest_fluxes ./= lya_absorption,
   rest_noise_variances ./= lya_absorption^2; then steps 3-4 as in training_set_oracle;
5'. the PCA starts from a copy of centered_rest_fluxes whose NaNs are replaced by each row's nanmedian, decomposed by
   pca(filled, 'rows', 'complete'): the covariance of the complete rows, which is ``pairwise_covariance`` of the filled
   matrix (an all-NaN row stays NaN and drops out of every pair and every column mean).

Restatement decisions, not pinned against MATLAB: the Lya term has no indicator; the noisy-pixel rule reads the noise
variance before the correction; an even count's median is MATLAB's meanof(a, b) = a + (b - a) / 2, or (a + b) / 2 when
sign(a) ~= sign(b) (sign(0) = 0) or either is infinite; eigh of the covariance stands for pca's SVD.
Pinned by the known-answer tests in tests/test_training_set_meanflux.py."""
import numpy as np

from . import process_qsos_multi_oracle as MO
from . import process_qsos_oracle as O
from .training_set_oracle import (centre, initial_x, interp_linear, lya_wavelength, nanstd, pairwise_covariance,
                                  pca_initial_M, rest_wavelengths)

max_noise_variance_multi = 3.0 ** 2                                          # set_parameters_multi.m:37
num_forest_lines = MO.num_forest_lines
all_transition_wavelengths = MO.all_transition_wavelengths                   # Angstrom
all_oscillator_strengths = MO.all_oscillator_strengths


def kim_tau():
    """prev_tau_0 f_l / f_lya * lambda_l / lya_wavelength, left to right as ...meanflux.m:271-273 (and the inference
    oracle) write it."""
    return np.array([MO.prev_tau_0 * all_oscillator_strengths[l] / MO.lya_oscillator_strength
                     * all_transition_wavelengths[l] / O.lya_wavelength for l in range(all_transition_wavelengths.size)])


def training_matrices_meanflux(wavelengths, flux, noise_variance, pixel_mask, z_qsos, rest,
                               max_nv=max_noise_variance_multi, num_forest_lines=num_forest_lines, lya=lya_wavelength):
    """Steps 1'-3' on ragged lists: (lya_1pzs, rest_fluxes, rest_noise_variances, lya_absorption), [N x P].  With
    num_forest_lines = 0 the absorption is 1 and the first three equal ``training_set_oracle.training_matrices`` bit for bit."""
    N, P = len(z_qsos), rest.size
    lya_1pzs, rest_fluxes, rest_nv = (np.full((N, P), np.nan) for _ in range(3))
    lya_absorption = np.ones((N, P))
    tau = kim_tau()
    for i in range(N):
        lam = np.asarray(wavelengths[i], dtype=np.float64)
        m = np.asarray(pixel_mask[i], dtype=bool)
        x = lam / (1.0 + z_qsos[i])
        f = np.where(m, np.nan, np.asarray(flux[i], dtype=np.float64))
        v = np.where(m, np.nan, np.asarray(noise_variance[i], dtype=np.float64))
        w = 1.0 + (lam - lya) / lya
        lya_1pzs[i] = interp_linear(x, w, rest)
        rest_fluxes[i] = interp_linear(x, f, rest)
        rest_nv[i] = interp_linear(x, v, rest)
        with np.errstate(invalid="ignore"):
            noisy = rest_nv[i] > max_nv                                      # step 2', before the correction
        lya_1pzs[i, noisy] = np.nan
        rest_fluxes[i, noisy] = np.nan
        rest_nv[i, noisy] = np.nan
        total = np.zeros(P)
        for l in range(num_forest_lines):                                    # step 3', ascending l
            wl = all_transition_wavelengths[l]
            one_plus_z = interp_linear(x, 1.0 + (lam - wl) / wl, rest)       # step 1': the same j and t as above
            one_plus_z[noisy] = np.nan
            with np.errstate(invalid="ignore"):
                term = tau[l] * one_plus_z ** MO.prev_beta
                if l > 0:
                    term = term * (one_plus_z <= 1.0 + z_qsos[i])            # value .* indicator: +0 or NaN
            total = np.where(np.isnan(term), total, total + term)             # nansum: NaN terms are skipped
        lya_absorption[i] = np.exp(-total)
    return lya_1pzs, rest_fluxes / lya_absorption, rest_nv / lya_absorption ** 2, lya_absorption


def matlab_meanof(a, b):
    """median.m's meanof for a <= b: a + (b - a) / 2, or (a + b) / 2 where sign(a) ~= sign(b) or either is infinite."""
    if np.sign(a) != np.sign(b) or np.isinf(a) or np.isinf(b):
        return (a + b) / 2
    return a + (b - a) / 2


def row_nanmedian(row):
    """nanmedian of one row: NaN for an all-NaN row, the middle value of an odd count, meanof of the middle two."""
    v = np.sort(row[~np.isnan(row)])
    n = v.size
    if n == 0:
        return np.nan
    if n % 2:
        return v[n // 2]
    return matlab_meanof(v[n // 2 - 1], v[n // 2])


def row_nanmedian_fill(X):
    """Step 5': a copy of X with each row's NaNs replaced by that row's nanmedian (all-NaN rows stay NaN)."""
    out = np.array(X, dtype=np.float64, copy=True)
    for i in range(out.shape[0]):
        nan = np.isnan(out[i])
        if nan.any():
            out[i, nan] = row_nanmedian(out[i])
    return out


def training_set_meanflux(spectra, k, rest=None, max_nv=max_noise_variance_multi, num_forest_lines=num_forest_lines,
                          fill=True):
    """Steps 1'-5' and 4, 6 on the ragged lists of preload_qsos plus z_qsos.  ``fill=False`` decomposes the pairwise
    covariance of the NaN matrix instead (learn_qso_model.m's start): with num_forest_lines = 0 and max_nv = 1 this is
    ``training_set_oracle.training_set``."""
    rest = rest_wavelengths() if rest is None else rest
    lya_1pzs, rest_fluxes, rest_nv, absorption = training_matrices_meanflux(
        spectra["all_wavelengths"], spectra["all_flux"], spectra["all_noise_variance"], spectra["all_pixel_mask"],
        np.asarray(spectra["z_qsos"], dtype=np.float64), rest, max_nv, num_forest_lines)
    mu, centered, num_observed = centre(rest_fluxes)
    std_dev = nanstd(centered)
    filled = row_nanmedian_fill(centered) if fill else centered
    C, counts = pairwise_covariance(filled)
    M, latent = pca_initial_M(C, k)
    return dict(rest_wavelengths=rest, lya_1pzs=lya_1pzs, centered_rest_fluxes=centered, rest_noise_variances=rest_nv,
                lya_absorption=absorption, mu=mu, num_observed=num_observed, std_dev=std_dev, filled=filled, cov=C,
                counts=counts, latent=latent, initial_x=initial_x(M, np.log(std_dev)))
