r"""TEST INFRASTRUCTURE (oracle): literal NumPy restatement of the training-set construction and PCA initialisation of
the reference's learn_qso_model.m:36-110, one spectrum at a time, in the operation order the CUDA kernels follow:

1. per spectrum (:36-64): emitted wavelengths x = lambda / (1 + z); flux and noise variance NaN where masked;
   w = 1 + (lambda - lya_wavelength) / lya_wavelength; w, flux and noise variance interpolated linearly onto the rest
   grid (interp1): NaN outside [x_0, x_{L-1}], j = the largest index with x_j <= r capped at L - 2,
   t = (r - x_j) / (x_{j+1} - x_j), v = v_j + t (v_{j+1} - v_j), each a separate IEEE operation; lengths < 2 -> NaN row;
2. noisy pixels (:66-69): interpolated noise variance > max_noise_variance -> NaN in all three matrices;
3. mu = nanmean of each rest-flux column, centered_rest_fluxes = rest_fluxes - mu (:71-75);
4. initial_log_omega = log(nanstd(centered_rest_fluxes)), n - 1 normalisation (:82-95);
5. pca(centered_rest_fluxes, 'rows', 'pairwise'): X~ = X - nanmean(X) again, C = X~0' X~0 / (M'M - 1) with X~0 = X~ with
   NaN -> 0 and M the observed mask (NaN where the pair count is < 2); eigenpairs in descending order, the largest |entry|
   of each eigenvector (first on ties) positive; initial_M = coeff(:, 1:k) * sqrt(latent(1:k));
6. initial_x = [initial_M(:); initial_log_omega; log 0.1; log 0.0023; log 3.65] (set_parameters.m:40-42);
7. unpacking after the fit (:101-110).

The interval search and formula are written out instead of np.interp, which special-cases exact knots and NaN slopes.
Parity unpinned against MATLAB outputs (no MATLAB, reference run or SDSS data in the image); two points are known to be
ours and not MATLAB's: the exact-knot case of interp1 (a grid point equal to an observed emitted wavelength) and the
rounding of pca's internal sums.  Pinned by the known-answer tests in tests/test_training_set.py."""
import numpy as np

lya_wavelength = 1215.6701          # set_parameters.m:5
max_noise_variance = 1.0 ** 2
initial_c_0, initial_tau_0, initial_beta = 0.1, 0.0023, 3.65


def rest_wavelengths(min_lambda=911.75, max_lambda=1215.75, dlambda=0.25):
    return min_lambda + dlambda * np.arange(int(round((max_lambda - min_lambda) / dlambda)) + 1)


def interp_linear(x, v, r):
    """interp1(x, v, r, 'linear') with NaN outside [x_0, x_{L-1}] (elementwise over the grid points)."""
    out = np.full(r.size, np.nan)
    L = x.size
    if L < 2:
        return out
    inside = (r >= x[0]) & (r <= x[L - 1])
    ri = r[inside]
    j = np.minimum(np.searchsorted(x, ri, side="right") - 1, L - 2)        # largest j with x_j <= r, capped
    t = (ri - x[j]) / (x[j + 1] - x[j])
    d = v[j + 1] - v[j]
    out[inside] = v[j] + t * d
    return out


def training_matrices(wavelengths, flux, noise_variance, pixel_mask, z_qsos, rest, max_nv=max_noise_variance,
                      lya=lya_wavelength):
    """Steps 1-2 on ragged lists: (lya_1pzs, rest_fluxes, rest_noise_variances), [N x P]."""
    N, P = len(z_qsos), rest.size
    lya_1pzs, rest_fluxes, rest_nv = (np.full((N, P), np.nan) for _ in range(3))
    for i in range(N):
        lam = np.asarray(wavelengths[i], dtype=np.float64)
        m = np.asarray(pixel_mask[i], dtype=bool)
        x = lam / (1.0 + z_qsos[i])                                           # :40
        f = np.where(m, np.nan, np.asarray(flux[i], dtype=np.float64))      # :44-45
        v = np.where(m, np.nan, np.asarray(noise_variance[i], dtype=np.float64))
        w = 1.0 + (lam - lya) / lya                                          # :52-54
        lya_1pzs[i] = interp_linear(x, w, rest)
        rest_fluxes[i] = interp_linear(x, f, rest)                           # :57-59
        rest_nv[i] = interp_linear(x, v, rest)                               # :62-64
    with np.errstate(invalid="ignore"):
        noisy = rest_nv > max_nv                                             # :66-69 (NaN > t is False)
    lya_1pzs[noisy] = np.nan
    rest_fluxes[noisy] = np.nan
    rest_nv[noisy] = np.nan
    return lya_1pzs, rest_fluxes, rest_nv


def centre(rest_fluxes):
    """Step 3: (mu, centered_rest_fluxes, num_observed)."""
    num_observed = np.count_nonzero(~np.isnan(rest_fluxes), axis=0)
    with np.errstate(invalid="ignore", divide="ignore"):
        mu = np.nansum(rest_fluxes, axis=0) / num_observed                   # :71
    return mu, rest_fluxes - mu[None, :], num_observed                      # :75


def nanstd(X):
    """Column standard deviation over the non-NaN entries about their own mean, n - 1 normalisation."""
    obs = ~np.isnan(X)
    n = obs.sum(axis=0)
    with np.errstate(invalid="ignore", divide="ignore"):
        m = np.nansum(X, axis=0) / n
        return np.sqrt(np.nansum((X - m[None, :]) ** 2, axis=0) / (n - 1))


def pairwise_covariance(X):
    """The covariance of pca(X, 'rows', 'pairwise'): (C, counts), NaN where a pair is observed fewer than 2 times."""
    obs = ~np.isnan(X)
    with np.errstate(invalid="ignore", divide="ignore"):
        Xt = X - (np.nansum(X, axis=0) / obs.sum(axis=0))[None, :]
    X0 = np.where(obs, Xt, 0.0)
    Mo = obs.astype(np.float64)
    counts = (Mo.T @ Mo).astype(np.int64)
    with np.errstate(invalid="ignore", divide="ignore"):
        C = (X0.T @ X0) / (counts - 1)
    C[counts < 2] = np.nan
    return C, counts


def pca_initial_M(C, k):
    """Step 5 from the covariance: (initial_M [P x k], latent [k]); descending eigenpairs, pca's sign convention."""
    latent, coeff = np.linalg.eigh(C)
    latent, coeff = latent[::-1], coeff[:, ::-1]
    for c in range(coeff.shape[1]):
        big = int(np.argmax(np.abs(coeff[:, c])))                            # first on ties
        if coeff[big, c] < 0:
            coeff[:, c] = -coeff[:, c]
    return coeff[:, :k] * np.sqrt(latent[:k])[None, :], latent


def initial_x(initial_M, initial_log_omega):
    """Step 6: the layout of objective.m / objective_oracle.objective."""
    return np.concatenate([initial_M.T.ravel(), initial_log_omega,
                           [np.log(initial_c_0), np.log(initial_tau_0), np.log(initial_beta)]])


def unpack(x, num_pixels, k):
    """Step 7 (learn_qso_model.m:101-110): M, log_omega, log_c_0, log_tau_0, log_beta."""
    M = x[:num_pixels * k].reshape(k, num_pixels).T
    return M, x[num_pixels * k:num_pixels * (k + 1)], x[-3], x[-2], x[-1]


def training_set(spectra, k, rest=None, max_nv=max_noise_variance):
    """Steps 1-6 on the ragged lists of preload_qsos plus z_qsos."""
    rest = rest_wavelengths() if rest is None else rest
    lya_1pzs, rest_fluxes, rest_nv = training_matrices(spectra["all_wavelengths"], spectra["all_flux"],
                                                       spectra["all_noise_variance"], spectra["all_pixel_mask"],
                                                       np.asarray(spectra["z_qsos"], dtype=np.float64), rest, max_nv)
    mu, centered, num_observed = centre(rest_fluxes)
    std_dev = nanstd(centered)
    C, counts = pairwise_covariance(centered)
    M, latent = pca_initial_M(C, k)
    return dict(rest_wavelengths=rest, lya_1pzs=lya_1pzs, centered_rest_fluxes=centered, rest_noise_variances=rest_nv,
                mu=mu, num_observed=num_observed, std_dev=std_dev, cov=C, counts=counts, latent=latent,
                initial_x=initial_x(M, np.log(std_dev)))
