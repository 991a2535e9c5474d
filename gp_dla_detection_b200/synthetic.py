"""Seeded synthetic DR12Q-shaped inputs for the hot path (SURVEY.md section 8(d)).

There is no network and no SDSS data in the image, so tests and ``bench.py`` draw a
random-init k-dimensional null model, quasi-Monte-Carlo DLA samples, a prior catalogue and
BOSS-grid spectra with the shapes the reference's ``preload_qsos.m`` / ``learn_qso_model.m`` /
``generate_dla_samples.m`` produce.  Data generation only -- nothing here is on the product path.
"""
from __future__ import annotations

import math

import numpy as np

from . import params as P

MODEL_SEED = 20160516
SPECTRA_SEED = 162861


def make_model(k: int = 20, seed: int = MODEL_SEED) -> dict:
    """Random-init null model on the reference grid 911.75:0.25:1215.75 (learn_qso_model.m:29)."""
    rng = np.random.default_rng(seed)
    n = int(round((P.DEFAULT.max_lambda - P.DEFAULT.min_lambda) / P.DEFAULT.dlambda)) + 1   # 1217
    lam = P.DEFAULT.min_lambda + P.DEFAULT.dlambda * np.arange(n)
    mu = 1.0 + 0.5 * np.exp(-0.5 * ((lam - 1215.67) / 15.0) ** 2) + 0.15 * np.exp(-0.5 * ((lam - 1025.72) / 10.0) ** 2)
    j = np.arange(k)
    M = 0.15 / np.sqrt(j + 1.0) * np.cos(math.pi * (j + 1.0) * (lam[:, None] - P.DEFAULT.min_lambda) / 304.0)
    M = M + 0.02 * rng.standard_normal((n, k))
    log_omega = np.log(0.08 + 0.04 * rng.random(n))
    return dict(rest_wavelengths=lam, mu=mu, M=np.ascontiguousarray(M), log_omega=log_omega,
                log_c_0=math.log(0.1), log_tau_0=math.log(0.0023), log_beta=math.log(3.65))


def _radical_inverse(i: np.ndarray, base: int) -> np.ndarray:
    out = np.zeros(i.shape, dtype=np.float64)
    f = 1.0 / base
    i = i.copy()
    while np.any(i > 0):
        out += f * (i % base)
        i //= base
        f /= base
    return out


def make_samples(num_dla_samples: int = 10000, with_lls: bool = False) -> dict:
    """Deterministic stand-in for generate_dla_samples.m:8-57: 2-D Halton (bases 2, 3), second
    dimension pushed through the inverse CDF of 0.9*p_fit + 0.1*U[20, 23] with the surrogate
    p_fit(x) ~ exp(-1.5 (x - 20)) on [20, 25) (the real quadratic fit needs the DLA catalogue)."""
    idx = np.arange(1, num_dla_samples + 1, dtype=np.int64)
    offset_samples = _radical_inverse(idx, 2)
    u = _radical_inverse(idx, 3)
    grid = np.linspace(20.0, 25.0, 200001)
    fit = np.exp(-1.5 * (grid - 20.0))
    fit /= np.trapezoid(fit, grid)
    pdf = 0.9 * fit + 0.1 * ((grid <= 23.0) / 3.0)
    cdf = np.concatenate([[0.0], np.cumsum(0.5 * (pdf[1:] + pdf[:-1]) * np.diff(grid))])
    cdf /= cdf[-1]
    log_nhi_samples = np.interp(u, cdf, grid)
    out = dict(offset_samples=offset_samples, log_nhi_samples=log_nhi_samples,
               nhi_samples=10.0 ** log_nhi_samples)
    if with_lls:   # multi_dlas/set_lls_parameters.m:55-63: uniform in log N on [19.5, 20)
        u3 = _radical_inverse(idx, 5)
        out["lls_log_nhi_samples"] = 19.5 + 0.5 * u3
        out["lls_nhi_samples"] = 10.0 ** out["lls_log_nhi_samples"]
        # partition functions of the column-density prior below / above 10^20 (set_lls_parameters.m:64-71);
        # surrogate values for the synthetic prior (flat extrapolation below 20)
        out["Z_lls"], out["Z_dla"] = 0.18, 0.82
    return out


def make_prior(num: int = 50000, seed: int = 7) -> dict:
    """Synthetic prior catalogue: z_qsos and DLA flags (process_qsos.m:11-13)."""
    rng = np.random.default_rng(seed)
    z = 2.15 + rng.gamma(2.0, 0.3, size=num)
    return dict(z_qsos=np.minimum(z, 5.5), dla_ind=rng.random(num) < 0.1)


def _voigt_raw(lam_obs: np.ndarray, z: float, nhi: float) -> np.ndarray:
    """Unconvolved Ly-alpha-only absorption used to inject a DLA into synthetic flux."""
    from scipy.special import wofz
    c, sigma = 2.99792458e10, 9.08537121627923800e5
    tw, gam = 1.2156701e-05, 6.06075804241938613e+02
    lc = math.pi * 4.803204672997660e-10 ** 2 * 0.4164 * tw / (9.10938356e-28 * c)
    v = lam_obs * (c / (tw * (1 + z)) / 1e8) - c
    V = wofz((v + 1j * gam) / (math.sqrt(2) * sigma)).real / (math.sqrt(2 * math.pi) * sigma)
    return np.exp(-nhi * lc * V)


# Lyman series (wavelength in Angstrom, oscillator strength) for the mean-flux suppression of the multi-DLA
# path (multi_dlas/set_parameters_multi.m:76-145)
_LYMAN_A = np.array([1.2156701e-05, 1.0257223e-05, 9.725368e-06, 9.497431e-06, 9.378035e-06, 9.307483e-06,
                     9.262257e-06, 9.231504e-06, 9.209631e-06, 9.193514e-06, 9.181294e-06, 9.171806e-06,
                     9.16429e-06, 9.15824e-06, 9.15329e-06, 9.14919e-06, 9.14576e-06, 9.14286e-06, 9.14039e-06,
                     9.13826e-06, 9.13641e-06, 9.13480e-06, 9.13339e-06, 9.13215e-06, 9.13104e-06, 9.13006e-06,
                     9.12918e-06, 9.12839e-06, 9.12768e-06, 9.12703e-06, 9.12645e-06]) * 1e8
_LYMAN_F = np.array([0.416400, 0.079120, 0.029000, 0.013940, 0.007799, 0.004814, 0.003183, 0.002216, 0.001605,
                     0.00120, 0.000921, 0.0007226, 0.000577, 0.000469, 0.000386, 0.000321, 0.000270, 0.000230,
                     0.000197, 0.000170, 0.000148, 0.000129, 0.000114, 0.000101, 0.000089, 0.000080, 0.000071,
                     0.000064, 0.000058, 0.000053, 0.000048])


def forest_suppression(lam: np.ndarray, z_qso: float, tau_0: float, beta: float):
    """(mean-flux absorption, effective optical depth for the noise scaling) of the Lyman-series forest,
    the model of multi_dlas/process_qsos_multiple_dlas_meanflux.m:243-285 (Kim et al. 2007 prior)."""
    lya_1pz = lam / P.lya_wavelength
    depth = tau_0 * lya_1pz ** beta
    total = 0.0023 * lya_1pz ** 3.65
    for l in range(1, _LYMAN_A.size):
        onepz = lam / _LYMAN_A[l]
        ok = onepz <= 1 + z_qso
        ratio = _LYMAN_A[l] * _LYMAN_F[l] / (_LYMAN_A[0] * _LYMAN_F[0])
        depth = depth + np.where(ok, tau_0 * ratio * onepz ** beta, 0.0)
        total = total + np.where(ok, 0.0023 * ratio * onepz ** 3.65, 0.0)
    return np.exp(-total), depth


def make_spectra(model: dict, num_quasars: int, seed: int = SPECTRA_SEED, shard: int = 0,
                 fixed_shape: bool = False, dla_fraction: float = 0.1, meanflux: bool = False,
                 max_injected: int = 1, second_dla_fraction: float = 0.0) -> dict:
    """BOSS-grid spectra shaped like preload_qsos.m:56-67 output (ragged lists).

    ``fixed_shape`` gives the 1217-pixel micro-benchmark variant of BASELINE.json: exactly
    n = n_u = 1217 consecutive unmasked pixels inside the modelled window.
    ``second_dla_fraction``: the fraction of spectra with an injected DLA that get a second one, at least
    kms_to_z(3000) from the first in z (the multi-DLA model's separation); its truth is in ``truth_z_dla2`` /
    ``truth_log_nhi2`` (NaN where there is none), keys present only when the fraction is positive.  At 0 the
    generator draws exactly the random numbers it draws without the option."""
    rng = np.random.default_rng(seed + shard)
    lam_rest, mu, M, log_omega = model["rest_wavelengths"], model["mu"], model["M"], model["log_omega"]
    c_0, tau_0, beta = math.exp(model["log_c_0"]), math.exp(model["log_tau_0"]), math.exp(model["log_beta"])
    k = M.shape[1]
    out = dict(all_wavelengths=[], all_flux=[], all_noise_variance=[], all_pixel_mask=[], z_qsos=[],
               truth_z_dla=[], truth_log_nhi=[])
    truth2 = ("truth_z_dla2", "truth_log_nhi2") if second_dla_fraction > 0 else ()
    for nm in truth2:
        out[nm] = []
    sep = P.kms_to_z(3000.0)
    while len(out["z_qsos"]) < num_quasars:
        z_qso = min(2.15 + rng.gamma(2.0, 0.3), 5.5)
        j0 = math.ceil((math.log10(P.DEFAULT.loading_min_lambda * (1 + z_qso)) - 3.5563) / 1e-4) - 1
        j1 = math.floor((math.log10(P.DEFAULT.loading_max_lambda * (1 + z_qso)) - 3.5563) / 1e-4) + 1
        lam = 10.0 ** (3.5563 + 1e-4 * np.arange(j0, j1 + 1))
        rest = lam / (1 + z_qso)
        if fixed_shape:
            inside = np.flatnonzero((rest >= P.DEFAULT.min_lambda) & (rest <= P.DEFAULT.max_lambda))
            lam, rest = lam[inside[:1217]], rest[inside[:1217]]
        L = lam.size
        rc = np.clip(rest, lam_rest[0], lam_rest[-1])
        jj = np.minimum(((rc - lam_rest[0]) / P.DEFAULT.dlambda).astype(np.int64), lam_rest.size - 2)
        tt = (rc - lam_rest[jj]) / P.DEFAULT.dlambda
        mu_i = mu[jj] + tt * (mu[jj + 1] - mu[jj])
        M_i = M[jj] + tt[:, None] * (M[jj + 1] - M[jj])
        om2 = np.exp(2 * (log_omega[jj] + tt * (log_omega[jj + 1] - log_omega[jj])))
        if meanflux:   # the multi-DLA path's null model: forest-suppressed mean flux, Lyman-series noise
            absorb, depth = forest_suppression(lam, z_qso, tau_0, beta)
            om2 = om2 * (1 - np.exp(-depth) + c_0) ** 2 * absorb ** 2
            mu_i, M_i = mu_i * absorb, M_i * absorb[:, None]
        else:
            om2 = om2 * (1 - np.exp(-tau_0 * (lam / P.lya_wavelength) ** beta) + c_0) ** 2
        noise_variance = (0.1 + 0.4 * rng.random(L)) ** 2
        flux = mu_i + M_i @ rng.standard_normal(k) + np.sqrt(om2) * rng.standard_normal(L)
        tz, tn = np.nan, np.nan
        if rng.random() < dla_fraction:
            zmin = max(lam.min() / P.lya_wavelength - 1, P.lyman_limit * (1 + z_qso) / P.lya_wavelength - 1 + P.DEFAULT.min_z_cut)
            zmax = lam.max() / P.lya_wavelength - 1 - P.DEFAULT.max_z_cut
            for _ in range(int(rng.integers(1, max_injected + 1))):   # truth_* keep the last injected system
                tz, tn = rng.uniform(zmin, zmax), rng.uniform(20.0, 22.0)
                flux = flux * _voigt_raw(lam, tz, 10.0 ** tn)
        tz2, tn2 = np.nan, np.nan
        if truth2 and np.isfinite(tz) and rng.random() < second_dla_fraction:
            below, above = max(tz - sep - zmin, 0.0), max(zmax - tz - sep, 0.0)   # [zmin, tz - sep] + [tz + sep, zmax]
            x = rng.uniform(0.0, below + above)
            tz2 = zmin + x if x < below else tz + sep + (x - below)
            tn2 = rng.uniform(20.0, 22.0)
            if below + above > 0:
                flux = flux * _voigt_raw(lam, tz2, 10.0 ** tn2)
            else:
                tz2, tn2 = np.nan, np.nan
        flux = flux + np.sqrt(noise_variance) * rng.standard_normal(L)
        mask = np.zeros(L, dtype=bool) if fixed_shape else (rng.random(L) < 0.02)
        inside = (rest >= P.DEFAULT.min_lambda) & (rest <= P.DEFAULT.max_lambda)
        if np.count_nonzero(inside & ~mask) < P.DEFAULT.min_num_pixels:
            continue
        out["all_wavelengths"].append(lam); out["all_flux"].append(flux)
        out["all_noise_variance"].append(noise_variance); out["all_pixel_mask"].append(mask)
        out["z_qsos"].append(z_qso); out["truth_z_dla"].append(tz); out["truth_log_nhi"].append(tn)
        if truth2:
            out["truth_z_dla2"].append(tz2); out["truth_log_nhi2"].append(tn2)
    for nm in ("z_qsos", "truth_z_dla", "truth_log_nhi") + truth2:
        out[nm] = np.asarray(out[nm])
    return out
