"""Training set of the multi-DLA (mean-flux) null model (multi_dlas/learn_qso_model_meanflux.m): oracle known answers
for the Lyman-series mean-flux correction and the row-median fill on CPU, argument checks of the C entries on CPU,
parity of the CUDA kernels against the oracle and the device chain preload -> training set -> objective_lyseries ->
L-BFGS -> process_qsos_multiple_dlas_meanflux on the GPU."""
import ctypes

import numpy as np
import pytest

from oracle import training_set_meanflux_oracle as MF
from oracle import training_set_oracle as TS

LYA = 1215.6701
LYB = 1025.7223
HAND_REST = 1000.0 + np.arange(11.0)


def one_spectrum(x, z, flux=None, nv=None, mask=None):
    """One spectrum with emitted wavelengths x at redshift z (observed = x (1 + z))."""
    x = np.asarray(x, dtype=np.float64)
    return dict(all_wavelengths=[x * (1.0 + z)], all_flux=[np.ones(x.size) if flux is None else flux],
                all_noise_variance=[np.full(x.size, 0.25) if nv is None else nv],
                all_pixel_mask=[np.zeros(x.size, dtype=bool) if mask is None else mask], z_qsos=np.array([z]))


def matrices(sp, rest, **kw):
    return MF.training_matrices_meanflux(sp["all_wavelengths"], sp["all_flux"], sp["all_noise_variance"],
                                         sp["all_pixel_mask"], sp["z_qsos"], rest, **kw)


def meanflux_spectra(n, k=20, seed=0):
    from gp_dla_detection_b200 import synthetic as syn
    model = syn.make_model(k)
    return model, syn.make_spectra(model, n, seed=seed, dla_fraction=0, meanflux=True)


def with_edge_cases(sp):
    """Append a length-0 and a length-1 spectrum and make a few pixels noisy (noise variance above 3^2)."""
    out = {k: list(v) for k, v in sp.items() if k.startswith("all_")}
    for q in range(0, len(out["all_noise_variance"]), 97):
        nv = out["all_noise_variance"][q].copy()
        nv[100:104] = 12.0
        out["all_noise_variance"][q] = nv
    lam = out["all_wavelengths"][0]
    out["all_wavelengths"] += [np.zeros(0), lam[500:501].copy()]
    out["all_flux"] += [np.zeros(0), np.ones(1)]
    out["all_noise_variance"] += [np.zeros(0), np.full(1, 0.1)]
    out["all_pixel_mask"] += [np.zeros(0, dtype=bool), np.zeros(1, dtype=bool)]
    out["z_qsos"] = np.concatenate([sp["z_qsos"], sp["z_qsos"][:2]])
    return out


# ---------------------------------------------------------------- CPU: oracle known answers
def test_one_line_by_hand():
    z = 1.0
    sp = one_spectrum(999.5 + 2.0 * np.arange(7), z, flux=np.arange(7.0) + 1.0)
    lya, f, nv, a = matrices(sp, HAND_REST, num_forest_lines=1)
    plain, fp, nvp = TS.training_matrices(sp["all_wavelengths"], sp["all_flux"], sp["all_noise_variance"],
                                          sp["all_pixel_mask"], sp["z_qsos"], HAND_REST, max_nv=9.0)
    expect = np.exp(-0.0023 * (2.0 * HAND_REST / LYA) ** 3.65)
    assert np.allclose(a[0], expect, rtol=1e-14, atol=0)
    assert np.array_equal(lya, plain)                                   # lya_1pzs is not corrected
    assert np.array_equal(f[0], fp[0] / a[0]) and np.array_equal(nv[0], nvp[0] / a[0] ** 2)


def test_only_the_members_below_the_quasar_count():
    z = 3.0
    rest = np.array([972.0, 1020.0, 1025.5, 1026.0, 1100.0, 1200.0])   # knots of the spectrum below: t = 0
    sp = one_spectrum(np.arange(960.0, 1210.0, 0.5), z)
    a = {nl: matrices(sp, rest, num_forest_lines=nl)[3][0] for nl in (1, 2, 3, 31)}
    lam_a, lam_b, lam_g = MF.all_transition_wavelengths[:3]
    tau = MF.kim_tau()
    lam = rest * (1 + z)
    opz_a, opz_b = 1.0 + (lam - lam_a) / lam_a, 1.0 + (lam - lam_b) / lam_b
    lya_term = tau[0] * opz_a ** 3.65
    # between Lyb and Lya: only the Lya term (1 + z_b > 1 + z_qso)
    between = rest > lam_b
    assert between.sum() == 3 and np.all(opz_b[between] > 1 + z)
    assert np.array_equal(a[31][between], a[1][between])
    assert np.allclose(a[1][between], np.exp(-lya_term[between]), rtol=1e-14, atol=0)
    # below Lyb (and above Lyg): the Lyb term exactly where 1 + z_b <= 1 + z_qso
    below = (rest < lam_b) & (rest > lam_g)
    assert below.sum() == 2 and np.all(opz_b[below] <= 1 + z)
    assert np.array_equal(a[31][below], a[2][below]) and np.all(a[2][below] < a[1][below])
    assert np.allclose(a[2][below], np.exp(-(lya_term[below] + tau[1] * opz_b[below] ** 3.65)), rtol=1e-14, atol=0)
    # below Lyg (above Lyd) the third member counts too, and no other
    assert a[3][0] < a[2][0] and a[31][0] == a[3][0]


def test_nan_terms_are_skipped_and_noisy_pixels_go_first():
    z = 4.0
    x = 1000.0 + np.arange(0.0, 40.0, 1.0)
    nv = np.full(x.size, 0.25)
    nv[10] = 8.0                                                        # below 3^2 before the correction, far above after
    nv[20] = 12.0                                                       # above 3^2: removed
    mask = np.zeros(x.size, dtype=bool)
    mask[30] = True
    sp = one_spectrum(x, z, nv=nv, mask=mask)
    rest = 990.0 + np.arange(0.0, 60.0, 1.0)                            # grid points beyond either end of the spectrum
    lya, f, v, a = matrices(sp, rest)
    outside = (rest < x[0]) | (rest > x[-1])
    noisy = rest == 1020.0
    # nansum of NaN terms only: exp(-0) = 1 where nothing is observed; never NaN
    assert not np.isnan(a).any()
    assert np.all(a[0][outside] == 1.0) and np.all(a[0][noisy] == 1.0)
    assert np.all(np.isnan(lya[0][outside | noisy])) and np.all(np.isnan(f[0][outside | noisy]))
    assert np.all(np.isnan(v[0][outside | noisy]))
    # a masked flux pixel: the absorption is still computed (lya_1pzs and every 1 + z_l are not masked)
    masked = (rest > 1029.0) & (rest < 1031.0)
    assert np.all(np.isnan(f[0][masked])) and np.all(a[0][masked] < 1.0)
    # the rule reads the noise variance before the correction: 8 stays, and is 8 / a^2 > 9 afterwards
    kept = rest == 1010.0
    assert np.isfinite(v[0][kept]).all() and v[0][kept][0] == 8.0 / a[0][kept][0] ** 2 and v[0][kept][0] > 9.0


def test_zero_lines_reproduce_the_plain_oracle():
    from test_training_set import hand_spectra
    sp = hand_spectra()
    for max_nv in (1.0, 9.0):
        lya, f, nv, a = matrices(sp, HAND_REST, max_nv=max_nv, num_forest_lines=0)
        ref = TS.training_matrices(sp["all_wavelengths"], sp["all_flux"], sp["all_noise_variance"],
                                   sp["all_pixel_mask"], sp["z_qsos"], HAND_REST, max_nv=max_nv)
        for got, want in zip((lya, f, nv), ref):
            assert np.array_equal(got, want, equal_nan=True)
        assert np.all(a == 1.0)


def test_zero_lines_and_pairwise_pca_reproduce_training_set():
    _, sp = meanflux_spectra(300, seed=5)
    ref = TS.training_set(sp, 4)
    got = MF.training_set_meanflux(sp, 4, max_nv=1.0, num_forest_lines=0, fill=False)
    for n in ("lya_1pzs", "centered_rest_fluxes", "rest_noise_variances", "mu", "num_observed", "std_dev", "cov",
              "counts", "latent", "initial_x"):
        assert np.array_equal(got[n], ref[n], equal_nan=True), n


# ---------------------------------------------------------------- CPU: the row-median fill
def test_median_known_answers():
    nan = np.nan
    X = np.array([[3.0, nan, 1.0, 2.0, nan],                # odd count: 2
                  [1.0, 4.0, nan, 2.0, 3.0],                # even, same sign: 2 + (3 - 2) / 2
                  [-0.1, nan, 0.7, nan, nan],               # even, mixed signs: (a + b) / 2
                  [nan, nan, nan, nan, nan],                # all NaN: stays NaN
                  [0.0, 2.0, nan, nan, nan],                # sign(0) = 0 differs from sign(2): (a + b) / 2
                  [5.0, 6.0, 7.0, 8.0, 9.0]])               # complete: unchanged
    out = MF.row_nanmedian_fill(X)
    assert np.array_equal(out[0], [3.0, 2.0, 1.0, 2.0, 2.0])
    assert np.array_equal(out[1], [1.0, 4.0, 2.5, 2.0, 3.0])
    assert (-0.1 + 0.7) / 2 != -0.1 + (0.7 + 0.1) / 2                   # the two formulas differ on this pair
    assert np.array_equal(out[2], [-0.1, 0.3, 0.7, 0.3, 0.3]) and out[2, 1] == (-0.1 + 0.7) / 2
    assert np.all(np.isnan(out[3]))
    assert np.array_equal(out[4], [0.0, 2.0, 1.0, 1.0, 1.0])
    assert np.array_equal(out[5], X[5])
    assert MF.matlab_meanof(2.0, 3.0) == 2.5 and MF.matlab_meanof(-np.inf, 1.0) == -np.inf
    assert np.isnan(X[0, 1])                                            # the input is not changed


def test_covariance_of_filled_rows_is_the_complete_row_covariance():
    rng = np.random.default_rng(6)
    X = rng.standard_normal((80, 12)) @ rng.standard_normal((12, 12)) + 2.0
    X[rng.random(X.shape) < 0.25] = np.nan
    X[[3, 17, 40]] = np.nan                                             # all-NaN rows drop out
    filled = MF.row_nanmedian_fill(X)
    C, counts = TS.pairwise_covariance(filled)
    complete = filled[~np.isnan(filled).any(axis=1)]
    assert complete.shape[0] == 77 and np.all(counts == 77)
    ref = np.cov(complete, rowvar=False)
    assert np.max(np.abs(C - ref)) <= 1e-13 * np.abs(ref).max()


# ---------------------------------------------------------------- CPU: recovery of a known model
@pytest.fixture(scope="module")
def recovery_case():
    model, sp = meanflux_spectra(2000, seed=11)
    rest = TS.rest_wavelengths()
    args = (sp["all_wavelengths"], sp["all_flux"], sp["all_noise_variance"], sp["all_pixel_mask"], sp["z_qsos"], rest)
    _, f, _, _ = MF.training_matrices_meanflux(*args)
    mu, centred, n = TS.centre(f)
    _, f_plain, _ = TS.training_matrices(*args)
    mu_plain, _, _ = TS.centre(f_plain)
    return model, rest, mu, TS.nanstd(centred), n, mu_plain


def test_corrected_mu_recovers_the_model_mean(recovery_case):
    model, _, mu, std_dev, n, _ = recovery_case
    sel = n >= 200
    assert sel.sum() > 1000
    z = np.abs(mu[sel] - model["mu"][sel]) / (std_dev[sel] / np.sqrt(n[sel]))
    assert z.max() < 5.0, z.max()


def test_uncorrected_mu_is_biased_low_in_the_forest(recovery_case):
    model, rest, _, _, _, mu_plain = recovery_case
    forest = rest < 1200.0
    assert np.median(mu_plain[forest] / model["mu"][forest]) < 0.9


def test_lyman_series_tables():
    from gp_dla_detection_b200 import params
    assert np.array_equal(params.all_transition_wavelengths, MF.all_transition_wavelengths)
    assert np.array_equal(params.all_oscillator_strengths, MF.all_oscillator_strengths)
    assert params.all_transition_wavelengths[0] == pytest.approx(1215.6701, abs=1e-9)     # Angstrom
    assert params.num_forest_lines == 31 and (params.prev_tau_0, params.prev_beta) == (0.0023, 3.65)
    assert params.MULTI.max_noise_variance == 9.0 and params.DEFAULT.max_noise_variance == 1.0
    assert params.MULTI.k == params.DEFAULT.k and params.MULTI.min_lambda == params.DEFAULT.min_lambda


# ---------------------------------------------------------------- CPU: argument checks before any launch
def _vp(a):
    return ctypes.c_void_p(a.ctypes.data)


def test_new_entries_reject_bad_arguments():
    from gp_dla_detection_b200 import _lib
    lib = _lib.load()
    N, L, P = 2, 8, 5
    W, F, V = np.ones((N, L)), np.ones((N, L)), np.ones((N, L))
    Mk = np.zeros((N, L), dtype=np.uint8)
    z = np.ones(N)
    rest = 1000.0 + np.arange(P, dtype=np.float64)
    outs = [np.empty((N, P)) for _ in range(4)] + [np.empty(P), np.empty(P), np.empty(P, dtype=np.int32)]

    def call(n=N, lmax=L, lengths=None, grid=rest, npix=P, nl=31, device=False):
        lengths = np.array([L, 3], dtype=np.int32) if lengths is None else lengths
        args = [n, lmax, _vp(W), _vp(F), _vp(V), _vp(Mk), _vp(lengths), _vp(z), _vp(grid), npix, LYA, 9.0, nl,
                *[_vp(o) for o in outs]]
        return lib.gpdla_training_set_lyseries_device(*args, None) if device else lib.gpdla_training_set_lyseries(*args)

    err = lambda: lib.gpdla_last_error(None).decode()
    for device in (False, True):
        assert call(n=-1, device=device) == _lib.GPDLA_ERR_INVALID
        assert call(lmax=0, device=device) == _lib.GPDLA_ERR_INVALID
        assert call(npix=0, device=device) == _lib.GPDLA_ERR_INVALID
        for nl in (-1, 32):
            assert call(nl=nl, device=device) == _lib.GPDLA_ERR_INVALID
            assert "num_forest_lines" in err()
    assert call(lengths=np.array([L + 1, 3], dtype=np.int32)) == _lib.GPDLA_ERR_INVALID
    assert "gpdla_training_set_lyseries: lengths[0]" in err() and "outside [0, L_max" in err()
    assert call(lengths=np.array([-1, 3], dtype=np.int32)) == _lib.GPDLA_ERR_INVALID
    assert call(grid=rest[::-1].copy()) == _lib.GPDLA_ERR_INVALID
    assert "strictly increasing" in err()
    nulls = [None] * 7
    assert lib.gpdla_training_set_lyseries(N, L, None, None, None, None, None, None, _vp(rest), P, LYA, 9.0, 31,
                                           *nulls) == _lib.GPDLA_ERR_INVALID
    assert lib.gpdla_training_set_lyseries_device(N, L, None, None, None, None, None, None, _vp(rest), P, LYA, 9.0, 31,
                                                  *nulls, None) == _lib.GPDLA_ERR_INVALID
    X, out = np.ones((4, 3)), np.empty((4, 3))
    for n, p in ((-1, 3), (4, 0), (4, 16385)):
        assert lib.gpdla_row_nanmedian_fill(n, p, _vp(X), _vp(out)) == _lib.GPDLA_ERR_INVALID
        assert lib.gpdla_row_nanmedian_fill_device(n, p, _vp(X), _vp(out), None) == _lib.GPDLA_ERR_INVALID
    assert lib.gpdla_row_nanmedian_fill(4, 3, None, _vp(out)) == _lib.GPDLA_ERR_INVALID
    assert lib.gpdla_row_nanmedian_fill(4, 3, _vp(X), None) == _lib.GPDLA_ERR_INVALID
    assert lib.gpdla_row_nanmedian_fill_device(4, 3, _vp(X), None, None) == _lib.GPDLA_ERR_INVALID


def test_python_layer_rejects_bad_arguments():
    from gp_dla_detection_b200 import api
    from test_training_set import hand_spectra
    sp = api.pad_spectra(hand_spectra())
    with pytest.raises(ValueError, match="lengths"):
        api.training_set_meanflux(dict(sp, lengths=sp["lengths"] + 100), 2)
    with pytest.raises(ValueError, match="num_forest_lines"):
        api.training_set_meanflux(sp, 2, num_forest_lines=32)
    with pytest.raises(ValueError, match="2-D"):
        api.row_nanmedian_fill(np.ones(4))


# ---------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def parity_case():
    model, sp = meanflux_spectra(2999, seed=21)
    sp = with_edge_cases(sp)                                            # 3 001 spectra
    from gp_dla_detection_b200 import api
    return model, sp, MF.training_set_meanflux(sp, 10), api.training_set_meanflux(sp, 10)


@pytest.mark.gpu
def test_training_set_meanflux_matches_oracle(parity_case):
    _, sp, ref, res = parity_case
    assert res["lya_1pzs"].shape == (3001, 1217)
    assert np.array_equal(res["rest_wavelengths"], ref["rest_wavelengths"])
    assert np.array_equal(res["lya_1pzs"], ref["lya_1pzs"], equal_nan=True)
    for n in ("centered_rest_fluxes", "rest_noise_variances", "lya_absorption"):
        assert np.array_equal(np.isnan(res[n]), np.isnan(ref[n])), n
    a, ar = res["lya_absorption"], ref["lya_absorption"]
    assert not np.isnan(ar).any() and ar.min() < 0.5
    assert np.max(np.abs(a - ar) / ar) <= 1e-14
    ok = ~np.isnan(ref["rest_noise_variances"])
    nv, nvr = res["rest_noise_variances"][ok], ref["rest_noise_variances"][ok]
    assert np.max(np.abs(nv - nvr) / nvr) <= 1e-14
    y, yr = res["centered_rest_fluxes"], ref["centered_rest_fluxes"]
    ok = ~np.isnan(yr)
    assert np.max(np.abs(y[ok] - yr[ok])) <= 1e-14 * np.abs(yr[ok]).max()
    assert np.max(np.abs(res["mu"] - ref["mu"]) / np.abs(ref["mu"])) < 1e-13
    assert np.max(np.abs(res["std_dev"] - ref["std_dev"]) / ref["std_dev"]) < 1e-13
    assert np.array_equal(res["num_observed"], ref["num_observed"])
    assert np.all(np.isnan(res["lya_1pzs"][-2:])) and np.all(np.isnan(y[-2:])) and np.all(a[-2:] == 1.0)
    # the noisy-pixel rule at 3^2: with it disabled, the grid points whose interpolated noise variance exceeds 9 are
    # exactly the ones the rule adds to the NaN pattern of lya_1pzs
    lya_loose, _, nv_loose, _ = MF.training_matrices_meanflux(
        sp["all_wavelengths"], sp["all_flux"], sp["all_noise_variance"], sp["all_pixel_mask"], sp["z_qsos"],
        ref["rest_wavelengths"], max_nv=np.inf, num_forest_lines=0)
    with np.errstate(invalid="ignore"):
        noisy = nv_loose > 9.0
    assert noisy.sum() >= 60                                              # every 97th spectrum has a noisy stretch
    assert np.array_equal(np.isnan(res["lya_1pzs"]), np.isnan(lya_loose) | noisy)
    assert np.all(np.isnan(y[noisy])) and np.all(res["lya_absorption"][noisy] == 1.0)


@pytest.mark.gpu
def test_indicator_boundary_matches_oracle():
    """Grid points at, and within 1e-13 of, the series members' wavelengths, each a knot of the spectrum: there
    1 + z_l sits on 1 + z_qso to rounding, and the kernel must take the oracle's decision for every member."""
    from gp_dla_detection_b200 import _lib
    lib = _lib.load()
    tw = MF.all_transition_wavelengths
    knots = np.concatenate([tw[1:12], tw[1:12] * (1 - 1e-13), tw[1:12] * (1 + 1e-13), np.arange(905.0, 1220.0, 0.7)])
    x = np.unique(knots)
    z = np.array([3.0, 2.5, 3.7])
    sp = dict(all_wavelengths=[x * (1 + q) for q in z], all_flux=[1.0 + 0.01 * np.arange(x.size)] * 3,
              all_noise_variance=[np.full(x.size, 0.25)] * 3, all_pixel_mask=[np.zeros(x.size, dtype=bool)] * 3,
              z_qsos=z)
    rest = x[(x > 911.0) & (x < 1216.0)]
    _, f_ref, nv_ref, a_ref = matrices(sp, rest)
    N, L, P = 3, x.size, rest.size
    W = np.ascontiguousarray(np.stack(sp["all_wavelengths"]))
    F, V = np.stack(sp["all_flux"]), np.stack(sp["all_noise_variance"])
    Mk = np.zeros((N, L), dtype=np.uint8)
    lengths = np.full(N, L, dtype=np.int32)
    outs = [np.empty((N, P)) for _ in range(4)] + [np.empty(P), np.empty(P), np.empty(P, dtype=np.int32)]
    assert lib.gpdla_training_set_lyseries(N, L, _vp(W), _vp(F), _vp(V), _vp(Mk), _vp(lengths), _vp(z), _vp(rest), P,
                                           LYA, 9.0, 31, *[_vp(o) for o in outs]) == 0
    a = outs[3]
    assert np.max(np.abs(a - a_ref) / a_ref) <= 1e-14
    # one Lyman-series term changes the absorption by far more than 1e-14: every decision was the oracle's
    smallest_term = MF.kim_tau()[11] * 3.0 ** 3.65
    assert smallest_term > 1e-7
    assert np.max(np.abs(outs[2] - nv_ref) / nv_ref) <= 1e-14


@pytest.mark.gpu
def test_median_fill_and_covariance_match_oracle(parity_case):
    from gp_dla_detection_b200 import api
    _, _, ref, res = parity_case
    y = res["centered_rest_fluxes"]
    filled = api.row_nanmedian_fill(y)
    assert np.array_equal(filled, MF.row_nanmedian_fill(y), equal_nan=True)
    assert np.array_equal(np.isnan(filled).all(axis=1), np.isnan(y).all(axis=1))
    assert not np.isnan(filled[~np.isnan(filled).all(axis=1)]).any()
    assert np.array_equal(api.row_nanmedian_fill(y), filled, equal_nan=True)          # the same bits on every call
    cov, counts = api.pairwise_covariance(filled)
    assert np.array_equal(counts, ref["counts"])
    assert np.max(np.abs(cov - ref["cov"])) <= 1e-12 * np.abs(ref["cov"]).max()
    # small shapes, complete and all-NaN rows, a row size that is a power of two, one past it, and one
    rng = np.random.default_rng(14)
    for N, P in ((1, 1), (5, 7), (40, 2048), (9, 2049), (3, 1217)):
        X = rng.standard_normal((N, P))
        X[rng.random(X.shape) < 0.3] = np.nan
        X[0] = np.nan
        if N > 2:
            X[1] = rng.standard_normal(P)
        assert np.array_equal(api.row_nanmedian_fill(X), MF.row_nanmedian_fill(X), equal_nan=True), (N, P)


@pytest.mark.gpu
def test_initial_x_matches_oracle(parity_case):
    _, _, ref, res = parity_case
    k, P = 10, 1217
    top = ref["latent"][:k + 1]
    assert np.all(-np.diff(top) / top[1:] >= 1e-3), -np.diff(top) / top[1:]
    x, xr = res["initial_x"], ref["initial_x"]
    assert x.size == xr.size == P * (k + 1) + 3
    assert np.max(np.abs(x[:P * k] - xr[:P * k])) <= 1e-9 * np.abs(xr[:P * k]).max()
    assert np.max(np.abs(x[P * k:] - xr[P * k:]) / np.abs(xr[P * k:])) <= 1e-9


@pytest.mark.gpu
def test_zero_lines_give_the_plain_training_set_bits(parity_case):
    """gpdla_training_set_lyseries with num_forest_lines = 0 against gpdla_training_set, and repeated calls."""
    from gp_dla_detection_b200 import _lib, api
    _, sp, _, res = parity_case
    lib = _lib.load()
    pad = api.pad_spectra(sp)
    W, F, V = (np.ascontiguousarray(pad[n], dtype=np.float64) for n in ("wavelengths", "flux", "noise_variance"))
    Mk = np.ascontiguousarray(pad["pixel_mask"], dtype=np.uint8)
    lengths = np.ascontiguousarray(pad["lengths"], dtype=np.int32)
    z = np.ascontiguousarray(pad["z_qsos"], dtype=np.float64)
    rest = api.rest_wavelengths()
    N, L = W.shape
    P = rest.size

    def outputs(n_abs):
        return [np.empty((N, P)) for _ in range(3 + n_abs)] + [np.empty(P), np.empty(P), np.empty(P, dtype=np.int32)]

    for max_nv in (1.0, 9.0):
        plain = outputs(0)
        assert lib.gpdla_training_set(N, L, _vp(W), _vp(F), _vp(V), _vp(Mk), _vp(lengths), _vp(z), _vp(rest), P, LYA,
                                      max_nv, *[_vp(o) for o in plain]) == 0
        for absorption in (True, False):
            ly = outputs(1)
            args = [_vp(o) for o in ly]
            if not absorption:
                args[3] = None
            assert lib.gpdla_training_set_lyseries(N, L, _vp(W), _vp(F), _vp(V), _vp(Mk), _vp(lengths), _vp(z),
                                                   _vp(rest), P, LYA, max_nv, 0, *args) == 0
            for got, want in zip(ly[:3] + ly[4:], plain):
                assert np.array_equal(got, want, equal_nan=True)
            if absorption:
                assert np.all(ly[3] == 1.0)
    again = api.training_set_meanflux(sp, 10)
    for n, v in res.items():
        assert np.array_equal(again[n], v, equal_nan=True), n


@pytest.mark.gpu
def test_device_chain_matches_host_entry():
    """Raw coadds -> preload_qsos_device -> training_set_meanflux_device -> TrainingObjective(num_forest_lines=31) on
    those CUDA tensors: the same bits as the host entry api.training_set_meanflux and api.objective_lyseries."""
    import torch
    from gp_dla_detection_b200 import api, params
    from test_training_set import make_raw
    rng = np.random.default_rng(12)
    raw, z = make_raw(48, 13, rng.uniform(3.0, 3.5, 48))
    pad = api._pad_raw(raw)
    t = {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in pad.items()}
    zt = torch.from_numpy(z).cuda()
    pre = api.preload_qsos_device(t["flux"], t["loglam"], t["ivar"], t["and_mask"], t["lengths"], zt)
    k = 10
    dev = api.training_set_meanflux_device(pre["wavelengths"], pre["flux"], pre["noise_variance"], pre["pixel_mask"],
                                           pre["lengths"], zt, k)
    assert dev["centered_rest_fluxes"].is_cuda and isinstance(dev["initial_x"], np.ndarray)
    host_in = dict(wavelengths=pre["wavelengths"].cpu().numpy(), flux=pre["flux"].cpu().numpy(),
                   noise_variance=pre["noise_variance"].cpu().numpy(), pixel_mask=pre["pixel_mask"].cpu().numpy(),
                   lengths=pre["lengths"].cpu().numpy(), z_qsos=z)
    assert host_in["lengths"].min() > 0
    host = api.training_set_meanflux(host_in, k)
    for n in ("lya_1pzs", "centered_rest_fluxes", "rest_noise_variances", "lya_absorption", "mu", "std_dev",
              "num_observed"):
        assert np.array_equal(dev[n].cpu().numpy(), host[n], equal_nan=True), n
    assert np.array_equal(dev["initial_x"], host["initial_x"])
    assert host["lya_absorption"].min() < 0.7
    tw, osc = params.all_transition_wavelengths, params.all_oscillator_strengths
    ev = api.TrainingObjective(dev["centered_rest_fluxes"], dev["lya_1pzs"], dev["rest_noise_variances"], k,
                               num_forest_lines=31, all_transition_wavelengths=tw, all_oscillator_strengths=osc)
    assert ev.y.data_ptr() == dev["centered_rest_fluxes"].data_ptr()               # kept without a copy
    f, g = ev(dev["initial_x"])
    ev.close()
    fh, gh = api.objective_lyseries(host["initial_x"], host["centered_rest_fluxes"], host["lya_1pzs"],
                                    host["rest_noise_variances"], 31, tw, osc)
    assert f == fh and np.array_equal(g, gh)
    assert np.isfinite(f) and np.all(np.isfinite(g))


@pytest.mark.gpu
def test_learn_qso_model_meanflux_from_spectra_end_to_end():
    from gp_dla_detection_b200 import api, params, synthetic as syn
    model, sp = meanflux_spectra(2000, seed=31)
    k = 20
    learned = api.learn_qso_model_meanflux_from_spectra(sp, k, max_iter=30)
    P = 1217
    assert learned["M"].shape == (P, k) and learned["mu"].shape == (P,) and learned["log_omega"].shape == (P,)
    for n in ("mu", "M", "log_omega"):
        assert np.all(np.isfinite(learned[n])), n
    assert all(np.isfinite(learned[n]) for n in ("log_c_0", "log_tau_0", "log_beta", "log_likelihood"))
    ts = api.training_set_meanflux(sp, k)
    assert np.array_equal(ts["initial_x"], learned["initial_x"]) and np.array_equal(ts["mu"], learned["mu"])
    f0, _ = api.objective_lyseries(ts["initial_x"], ts["centered_rest_fluxes"], ts["lya_1pzs"],
                                   ts["rest_noise_variances"], 31, params.all_transition_wavelengths,
                                   params.all_oscillator_strengths)
    assert learned["log_likelihood"] < f0
    n = ts["num_observed"]
    sel = n >= 200
    assert sel.sum() > 1000
    zscore = np.abs(learned["mu"][sel] - model["mu"][sel]) / (ts["std_dev"][sel] / np.sqrt(n[sel]))
    assert zscore.max() < 5.0, zscore.max()
    samples, prior = syn.make_samples(2000, with_lls=True), syn.make_prior(2000)
    spectra = syn.make_spectra(syn.make_model(k), 4, seed=5, dla_fraction=0.5, meanflux=True)
    out = api.process_qsos_multiple_dlas_meanflux(learned, samples, spectra, prior, return_samples=False)
    for name in ("model_posteriors", "p_dlas", "p_no_dlas", "log_likelihoods_no_dla"):
        assert np.all(np.isfinite(out[name])), name
