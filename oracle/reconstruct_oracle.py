"""Literal CPU restatement of the fitted model of one quasar under chosen absorbers (test oracle).

TEST INFRASTRUCTURE ONLY -- see ``oracle/__init__.py``.  parity unpinned: the reference draws the fitted model on the
host in ``CDDF_analysis/qso_loader.py:1654-1774`` (``plot_this_mu``), which is not in this tree.  Built from the other
oracles: ``voigt``, ``padded_wavelengths`` and the interpolation of ``process_qsos_oracle`` (process_qsos.m:138-146,
168-176), ``suppressed_model`` of ``process_qsos_multi_oracle`` (...meanflux.m:245-293).  Restatement decisions (the
reference does not pin them):

* the planes cover the modelled window (``min_lambda <= lambda / (1 + z_qso) <= max_lambda``) only, masked pixels
  included; masked pixels get model values but no ``prior_sd`` (their noise variance is not used anywhere);
* absorbers multiply as instrument-convolved profiles, in the given order (...meanflux.m:342-351);
* ``continuum`` is the emitted continuum ``mu + M x^``, without the mean-flux suppression and the absorbers.

For the used pixels (window, not masked), with ``a`` the absorption:
``d = a^2 om2~ + v``, ``r = y - a mu~``, ``B = I + (aM~)' D^-1 (aM~)``, ``g = (aM~)' D^-1 r``, ``x^ = B^-1 g``,
``chi2 = sum r^2/d - g' B^-1 g``, ``log p = -1/2 (chi2 + sum log d + 2 sum log L_ii + n log 2 pi)`` (B = L L').
"""
from __future__ import annotations

import math

import numpy as np
from scipy.linalg import cho_solve, cholesky, solve_triangular

from . import process_qsos_multi_oracle as MO
from . import process_qsos_oracle as O

PLANES = ("absorption", "prior_mean", "prior_sd", "fit_mean", "continuum", "continuum_sd")


def woodbury(aM, d, r):
    """The low-rank Gaussian quantities of ``N(r; 0, aM aM' + diag(d))`` (log_mvnpdf_low_rank.m:5-34) in Woodbury
    form: ``B``, its lower Cholesky factor, ``x^ = B^-1 g``, ``chi2``, ``B^-1`` and the log-density."""
    n, k = aM.shape
    D_inv_M = aM / d[:, None]
    B = aM.T @ D_inv_M
    B[np.diag_indices(k)] += 1.0
    L = cholesky(B, lower=True)
    g = D_inv_M.T @ r
    x = cho_solve((L, True), g)
    chi2 = np.sum(r * r / d) - g @ x
    Linv = solve_triangular(L, np.eye(k), lower=True)
    B_inv = Linv.T @ Linv
    log_likelihood = -0.5 * (chi2 + np.sum(np.log(d)) + 2.0 * np.sum(np.log(np.diag(L))) + n * O.LOG_2PI)
    return dict(B=B, L=L, latent=x, chi2=chi2, B_inv=B_inv, log_likelihood=log_likelihood)


def window_model(model, this_wavelengths, this_rest_wavelengths, z_qso, meanflux):
    """(mu, M) unsuppressed and (mu~, M~, om2~) as the path being reconstructed evaluates them, on given pixels."""
    rest_wavelengths = model["rest_wavelengths"]
    this_mu = np.interp(this_rest_wavelengths, rest_wavelengths, model["mu"])                    # process_qsos.m:138
    this_M = np.stack([np.interp(this_rest_wavelengths, rest_wavelengths, model["M"][:, j])
                       for j in range(model["M"].shape[1])], axis=1)                             # :139
    if meanflux:
        mu_t, M_t, om2_t = MO.suppressed_model(model, this_wavelengths, this_rest_wavelengths, z_qso)
        return this_mu, this_M, mu_t, M_t, om2_t
    c_0, tau_0, beta = math.exp(model["log_c_0"]), math.exp(model["log_tau_0"]), math.exp(model["log_beta"])
    this_omega2 = np.exp(2.0 * np.interp(this_rest_wavelengths, rest_wavelengths, model["log_omega"]))   # :141-142
    this_lya_zs = (this_wavelengths - O.lya_wavelength) / O.lya_wavelength                      # :117-119
    this_scaling_factor = 1.0 - np.exp(-tau_0 * (1.0 + this_lya_zs) ** beta) + c_0              # :144
    return this_mu, this_M, this_mu, this_M, this_omega2 * this_scaling_factor ** 2             # :146


def reconstruct_one(model, wavelengths, flux, noise_variance, pixel_mask, z_qso, absorber_z=(), absorber_nhi=(),
                    meanflux=False, num_lines=O.num_lines_default):
    """One quasar: planes over its pixels (NaN outside the window), ``latent``, ``chi2``, ``log_likelihood``,
    ``num_pixels``, and the Woodbury quantities (``B``, ``B_inv``) for the checks."""
    this_wavelengths = np.asarray(wavelengths, dtype=np.float64)
    this_pixel_mask = np.asarray(pixel_mask).astype(bool)
    this_flux = np.asarray(flux, dtype=np.float64)
    this_noise_variance = np.asarray(noise_variance, dtype=np.float64)
    k = model["M"].shape[1]
    L = this_wavelengths.size
    out = {nm: np.full(L, np.nan) for nm in PLANES}
    out.update(latent=np.full(k, np.nan), chi2=np.nan, log_likelihood=np.nan, num_pixels=0)
    this_rest_wavelengths = this_wavelengths / (1.0 + z_qso)                                     # :102
    win = (this_rest_wavelengths >= O.min_lambda) & (this_rest_wavelengths <= O.max_lambda)     # :104-105
    used_all = win & ~this_pixel_mask                                                            # :110
    n = int(np.count_nonzero(used_all))
    if n == 0:                                                                                   # :74-82
        return out
    w_win = this_wavelengths[win]
    mu, M, mu_t, M_t, om2_t = window_model(model, w_win, this_rest_wavelengths[win], z_qso, meanflux)
    absorption = np.ones(w_win.size)
    padded = O.padded_wavelengths(w_win)                                                         # :168-176
    for z, N in zip(np.ravel(absorber_z), np.ravel(absorber_nhi)):
        if np.isnan(z):
            continue
        absorption = absorption * O.voigt(padded, z, N, num_lines)                               # ...meanflux.m:342-351
    used = ~this_pixel_mask[win]                                                                 # :181
    a_u = absorption[used]
    y, v = this_flux[win][used], this_noise_variance[win][used]
    d = om2_t[used] * a_u ** 2 + v
    r = y - mu_t[used] * a_u
    aM = M_t[used] * a_u[:, None]
    wb = woodbury(aM, d, r)
    x = wb["latent"]
    out.update(latent=x, chi2=wb["chi2"], log_likelihood=wb["log_likelihood"], num_pixels=n, B=wb["B"],
               B_inv=wb["B_inv"])
    prior_sd = np.sqrt(absorption ** 2 * (np.sum(M_t ** 2, axis=1) + om2_t) + this_noise_variance[win])
    prior_sd[~used] = np.nan
    planes = dict(absorption=absorption, prior_mean=absorption * mu_t, prior_sd=prior_sd,
                  fit_mean=absorption * (mu_t + M_t @ x), continuum=mu + M @ x,
                  continuum_sd=np.sqrt(np.sum((M @ wb["B_inv"]) * M, axis=1)))
    for nm in PLANES:
        out[nm][win] = planes[nm]
    return out


def reconstruct(model, spectra, absorber_z=None, absorber_nhi=None, meanflux=False, num_lines=O.num_lines_default,
                L_max=None):
    """Every quasar of ragged ``spectra`` (``all_wavelengths`` ... and ``z_qsos``): planes [Q, L_max] (NaN past each
    length), ``latent`` [Q, k], ``chi2``, ``log_likelihood``, ``num_pixels`` [Q]."""
    Q = len(spectra["z_qsos"])
    k = model["M"].shape[1]
    lengths = [len(w) for w in spectra["all_wavelengths"]]
    L_max = max(max(lengths) if Q else 1, 1) if L_max is None else L_max
    res = {nm: np.full((Q, L_max), np.nan) for nm in PLANES}
    res.update(latent=np.full((Q, k), np.nan), chi2=np.full(Q, np.nan), log_likelihood=np.full(Q, np.nan),
               num_pixels=np.zeros(Q, dtype=np.int32))
    for q in range(Q):
        az = () if absorber_z is None else np.atleast_2d(np.asarray(absorber_z, dtype=np.float64).reshape(Q, -1))[q]
        an = () if absorber_nhi is None else np.atleast_2d(np.asarray(absorber_nhi, dtype=np.float64).reshape(Q, -1))[q]
        o = reconstruct_one(model, spectra["all_wavelengths"][q], spectra["all_flux"][q],
                            spectra["all_noise_variance"][q], spectra["all_pixel_mask"][q], float(spectra["z_qsos"][q]),
                            az, an, meanflux, num_lines)
        for nm in PLANES:
            res[nm][q, :lengths[q]] = o[nm]
        for nm in ("latent", "chi2", "log_likelihood", "num_pixels"):
            res[nm][q] = o[nm]
    return res
