"""Training set and PCA initialisation of the null model (learn_qso_model.m:36-110): oracle known answers on CPU,
argument checks of the C entries on CPU, parity of the CUDA kernels against the oracle and the device chain
preload -> training set -> objective -> L-BFGS -> DLAProcessor on the GPU."""
import ctypes

import numpy as np
import pytest

from oracle import training_set_oracle as TS

LYA = 1215.6701


# ---------------------------------------------------------------- fixtures
def hand_spectra():
    """Four spectra on the grid 1000:1:1010 (rest), z = 1 (emitted wavelength = observed / 2, exact):
    0: x = 999.5:2:1011.5, flux j, noise variance 0.25, pixel 3 (x = 1005.5) masked;
    1: x = 1002.25:1:1006.25, noise variance 3 at x = 1004.25 (interpolates above 1 at r = 1004, 1005);
    2: one pixel; 3: no pixel."""
    x0 = 999.5 + 2.0 * np.arange(7)
    m0 = np.zeros(7, dtype=bool); m0[3] = True
    x1 = 1002.25 + np.arange(5.0)
    nv1 = np.array([0.5, 0.5, 3.0, 0.5, 0.5])
    return dict(all_wavelengths=[2 * x0, 2 * x1, np.array([2 * 1003.0]), np.zeros(0)],
                all_flux=[np.arange(7.0), np.array([1.0, 2.0, 3.0, 4.0, 5.0]), np.array([1.0]), np.zeros(0)],
                all_noise_variance=[np.full(7, 0.25), nv1, np.array([0.25]), np.zeros(0)],
                all_pixel_mask=[m0, np.zeros(5, dtype=bool), np.zeros(1, dtype=bool), np.zeros(0, dtype=bool)],
                z_qsos=np.array([1.0, 1.0, 1.0, 1.0]))


HAND_REST = 1000.0 + np.arange(11.0)


def synthetic_training_spectra(n, k=20, seed=0):
    from gp_dla_detection_b200 import synthetic as syn
    model = syn.make_model(k)
    return model, syn.make_spectra(model, n, seed=seed, dla_fraction=0)


def with_edge_cases(sp):
    """Append a length-0 and a length-1 spectrum and make a few pixels noisy (noise variance above 1)."""
    out = {k: list(v) for k, v in sp.items() if k.startswith("all_")}
    for q in range(0, len(out["all_noise_variance"]), 97):
        nv = out["all_noise_variance"][q].copy()
        nv[100:104] = 2.5
        out["all_noise_variance"][q] = nv
    lam = out["all_wavelengths"][0]
    out["all_wavelengths"] += [np.zeros(0), lam[500:501].copy()]
    out["all_flux"] += [np.zeros(0), np.ones(1)]
    out["all_noise_variance"] += [np.zeros(0), np.full(1, 0.1)]
    out["all_pixel_mask"] += [np.zeros(0, dtype=bool), np.zeros(1, dtype=bool)]
    out["z_qsos"] = np.concatenate([sp["z_qsos"], sp["z_qsos"][:2]])
    return out


def make_raw(Q, seed, z):
    """SDSS-like coadds on the BOSS grid (the columns preload_qsos reads)."""
    rng = np.random.default_rng(seed)
    raw = dict(flux=[], loglam=[], ivar=[], and_mask=[])
    for q in range(Q):
        n = int(rng.integers(4400, 4650))
        raw["loglam"].append(3.5563 + 1e-4 * (np.arange(n) + int(rng.integers(0, 30))))
        raw["flux"].append(3.0 + rng.standard_normal(n))
        ivar = rng.uniform(2.0, 8.0, n)
        ivar[rng.random(n) < 0.03] = 0.0
        raw["ivar"].append(ivar)
        am = np.zeros(n, dtype=np.int64)
        am[rng.random(n) < 0.02] |= 1 << 23
        raw["and_mask"].append(am)
    return raw, np.asarray(z, dtype=np.float64)


# ---------------------------------------------------------------- CPU: oracle known answers
def test_oracle_interpolation_known_answers():
    sp = hand_spectra()
    lya, f, nv = TS.training_matrices(sp["all_wavelengths"], sp["all_flux"], sp["all_noise_variance"],
                                      sp["all_pixel_mask"], sp["z_qsos"], HAND_REST)
    r = HAND_REST
    # spectrum 0: flux (r - 999.5) / 2 on the unmasked intervals; the masked pixel x = 1005.5 NaNs exactly the grid points
    # of its two adjacent intervals [1003.5, 1007.5]
    masked = (r > 1003.5) & (r < 1007.5)
    assert np.array_equal(np.isnan(f[0]), masked) and np.array_equal(np.isnan(nv[0]), masked)
    assert np.array_equal(f[0][~masked], (r[~masked] - 999.5) / 2)
    assert np.all(nv[0][~masked] == 0.25)
    assert np.all(np.isfinite(lya[0]))                                  # lya_1pzs is not masked (:52-54)
    assert np.allclose(lya[0], 2 * r / LYA, rtol=1e-15, atol=0)
    # spectrum 1: grid points beyond either end are NaN; the noisy pixel NaNs r = 1004, 1005 in all three matrices
    assert np.all(np.isnan(lya[1][(r < 1002.25) | (r > 1006.25)]))
    noisy = (r == 1004) | (r == 1005)
    inside = (r >= 1003) & (r <= 1006)
    assert np.all(np.isnan(lya[1][noisy])) and np.all(np.isnan(f[1][noisy])) and np.all(np.isnan(nv[1][noisy]))
    assert np.all(np.isfinite(lya[1][inside & ~noisy]))
    assert np.array_equal(f[1][inside & ~noisy], [1.75, 4.75])            # 1 + 0.75, 4 + 0.75
    assert np.array_equal(nv[1][inside & ~noisy], [0.5, 0.5])
    # the interpolated noise variances that trip the rule: 0.5 + 0.75 * 2.5 and 3 - 0.75 * 2.5
    _, _, nv_loose = TS.training_matrices(sp["all_wavelengths"], sp["all_flux"], sp["all_noise_variance"],
                                          sp["all_pixel_mask"], sp["z_qsos"], HAND_REST, max_nv=10.0)
    assert np.array_equal(nv_loose[1][noisy], [2.375, 1.125])
    # lengths 1 and 0: all-NaN rows
    for q in (2, 3):
        assert np.all(np.isnan(lya[q])) and np.all(np.isnan(f[q])) and np.all(np.isnan(nv[q]))


def test_oracle_exact_knots_and_ends():
    x = np.array([1.0, 2.0, 4.0])
    v = np.array([10.0, 20.0, 40.0])
    out = TS.interp_linear(x, v, np.array([0.5, 1.0, 2.0, 3.0, 4.0, 4.5]))
    # r = x_0: j = 0, t = 0; r = x_1: j = 1, t = 0; r = x_{L-1}: j capped at L - 2, t = 1
    assert np.array_equal(out, [np.nan, 10.0, 20.0, 30.0, 40.0, np.nan], equal_nan=True)
    out = TS.interp_linear(x, np.array([10.0, np.nan, 40.0]), np.array([1.0, 1.5, 2.0, 3.0]))
    assert np.all(np.isnan(out))                                        # a NaN at either end of the interval


def test_pairwise_covariance_oracle():
    rng = np.random.default_rng(3)
    X = rng.standard_normal((60, 9)) @ rng.standard_normal((9, 9))
    C, counts = TS.pairwise_covariance(X)
    assert np.max(np.abs(C - np.cov(X, rowvar=False))) < 1e-13 * np.abs(C).max()
    assert np.all(counts == 60)
    # with NaNs: a brute-force loop over the pairs, recentred by the column nanmeans
    X = rng.standard_normal((40, 12)) + 3.0
    X[rng.random(X.shape) < 0.3] = np.nan
    X[:, 7] = np.nan; X[[2, 5], 7] = [1.0, 2.0]                          # a column observed twice
    X[:, 8] = np.nan; X[11, 8] = 4.0                                    # and one observed once
    C, counts = TS.pairwise_covariance(X)
    m = np.nanmean(X, axis=0)
    for p in range(12):
        for q in range(12):
            both = ~np.isnan(X[:, p]) & ~np.isnan(X[:, q])
            n = int(both.sum())
            assert counts[p, q] == n
            if n < 2:
                assert np.isnan(C[p, q])
            else:
                ref = np.sum((X[both, p] - m[p]) * (X[both, q] - m[q])) / (n - 1)
                assert abs(C[p, q] - ref) <= 1e-14 * max(1.0, abs(ref)), (p, q)


def test_pca_sign_convention_and_layout():
    from oracle import objective_oracle as OB
    rng = np.random.default_rng(4)
    P, k = 30, 4
    A = rng.standard_normal((200, P)) @ rng.standard_normal((P, P))
    C = np.cov(A, rowvar=False)
    M, latent = TS.pca_initial_M(C, k)
    assert np.all(np.diff(latent) <= 0)
    coeff = M / np.sqrt(latent[:k])
    for c in range(k):
        assert coeff[np.argmax(np.abs(coeff[:, c])), c] > 0
        w, V = np.linalg.eigh(C)
        ref = V[:, -1 - c] * np.sign(V[np.argmax(np.abs(V[:, -1 - c])), -1 - c])
        assert np.allclose(coeff[:, c], ref, atol=1e-12)
    lw = np.log(np.sqrt(np.diag(C)))
    x = TS.initial_x(M, lw)
    assert x.size == P * (k + 1) + 3
    Mu, lwu, c0, t0, b = TS.unpack(x, P, k)
    assert np.array_equal(Mu, M) and np.array_equal(lwu, lw)
    assert (c0, t0, b) == (np.log(0.1), np.log(0.0023), np.log(3.65))
    # objective_oracle.objective reads the same layout: M = x[:P k].reshape(k, P).T
    y = rng.standard_normal((3, P)) * 0.3
    lya = np.full((3, P), 3.0)
    nv = np.full((3, P), 0.05)
    f, g = OB.objective(x, y, lya, nv)
    assert np.isfinite(f) and g.size == x.size


def test_oracle_mu_recovers_the_model_mean():
    model, sp = synthetic_training_spectra(2000, seed=11)
    out = TS.training_set(sp, 10)
    n = out["num_observed"]
    se = out["std_dev"] / np.sqrt(n)
    sel = n >= 200
    assert sel.sum() > 1000
    z = np.abs(out["mu"][sel] - model["mu"][sel]) / se[sel]
    assert z.max() < 5.0, z.max()
    assert out["initial_x"].size == 1217 * 11 + 3 and np.all(np.isfinite(out["initial_x"]))


def test_parameters_defaults():
    from gp_dla_detection_b200.params import Parameters
    p = Parameters()
    assert (p.max_noise_variance, p.initial_c_0, p.initial_tau_0, p.initial_beta) == (1.0, 0.1, 0.0023, 3.65)
    assert (p.min_lambda, p.max_lambda, p.dlambda, p.k) == (911.75, 1215.75, 0.25, 20)


# ---------------------------------------------------------------- CPU: argument checks before any launch
def _vp(a):
    return ctypes.c_void_p(a.ctypes.data)


def test_training_set_entry_rejects_bad_arguments():
    from gp_dla_detection_b200 import _lib
    lib = _lib.load()
    N, L, P = 2, 8, 5
    W, F, V = np.ones((N, L)), np.ones((N, L)), np.ones((N, L))
    Mk = np.zeros((N, L), dtype=np.uint8)
    z = np.ones(N)
    rest = 1000.0 + np.arange(P, dtype=np.float64)
    outs = [np.empty((N, P)) for _ in range(3)] + [np.empty(P), np.empty(P), np.empty(P, dtype=np.int32)]

    def call(n=N, lmax=L, lengths=None, grid=rest, npix=P):
        lengths = np.array([L, 3], dtype=np.int32) if lengths is None else lengths
        return lib.gpdla_training_set(n, lmax, _vp(W), _vp(F), _vp(V), _vp(Mk), _vp(lengths), _vp(z), _vp(grid), npix,
                                      LYA, 1.0, *[_vp(o) for o in outs])

    assert call(n=-1) == _lib.GPDLA_ERR_INVALID
    assert call(lmax=0) == _lib.GPDLA_ERR_INVALID
    assert call(npix=0) == _lib.GPDLA_ERR_INVALID
    assert call(lengths=np.array([L + 1, 3], dtype=np.int32)) == _lib.GPDLA_ERR_INVALID
    assert "outside [0, L_max" in lib.gpdla_last_error(None).decode()
    assert call(lengths=np.array([-1, 3], dtype=np.int32)) == _lib.GPDLA_ERR_INVALID
    assert call(grid=rest[::-1].copy()) == _lib.GPDLA_ERR_INVALID
    assert "strictly increasing" in lib.gpdla_last_error(None).decode()
    nulls = [None] * 6
    assert lib.gpdla_training_set(N, L, None, None, None, None, None, None, _vp(rest), P, LYA, 1.0,
                                  *nulls) == _lib.GPDLA_ERR_INVALID
    assert lib.gpdla_training_set_device(N, L, None, None, None, None, None, None, _vp(rest), P, LYA, 1.0,
                                         *nulls, None) == _lib.GPDLA_ERR_INVALID
    X = np.ones((4, 3))
    cov, cnt = np.empty((3, 3)), np.empty((3, 3), dtype=np.int32)
    assert lib.gpdla_pairwise_covariance(4, 0, _vp(X), _vp(cov), _vp(cnt)) == _lib.GPDLA_ERR_INVALID
    assert lib.gpdla_pairwise_covariance(-1, 3, _vp(X), _vp(cov), _vp(cnt)) == _lib.GPDLA_ERR_INVALID
    assert lib.gpdla_pairwise_covariance(4, 3, None, _vp(cov), _vp(cnt)) == _lib.GPDLA_ERR_INVALID
    assert lib.gpdla_pairwise_covariance_device(4, 3, _vp(X), None, _vp(cnt), None) == _lib.GPDLA_ERR_INVALID


def test_python_layer_rejects_bad_planes():
    from gp_dla_detection_b200 import api
    sp = api.pad_spectra(hand_spectra())
    bad = dict(sp, lengths=sp["lengths"] + 100)
    with pytest.raises(ValueError, match="lengths"):
        api.training_set(bad, 2)
    bad = dict(sp, z_qsos=sp["z_qsos"][:2])
    with pytest.raises(ValueError):
        api.training_set(bad, 2)


# ---------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def parity_case():
    model, sp = synthetic_training_spectra(2999, seed=21)
    sp = with_edge_cases(sp)                                            # 3 001 spectra
    from gp_dla_detection_b200 import api
    return model, sp, TS.training_set(sp, 10), api.training_set(sp, 10)


@pytest.mark.gpu
def test_training_set_matches_oracle(parity_case):
    _, sp, ref, res = parity_case
    assert res["lya_1pzs"].shape == (3001, 1217)
    assert np.array_equal(res["rest_wavelengths"], ref["rest_wavelengths"])
    assert np.array_equal(res["lya_1pzs"], ref["lya_1pzs"], equal_nan=True)
    assert np.array_equal(res["rest_noise_variances"], ref["rest_noise_variances"], equal_nan=True)
    y, yr = res["centered_rest_fluxes"], ref["centered_rest_fluxes"]
    assert np.array_equal(np.isnan(y), np.isnan(yr))
    ok = ~np.isnan(yr)
    assert np.max(np.abs(y[ok] - yr[ok])) <= 1e-13 * np.abs(yr[ok]).max()
    assert np.max(np.abs(res["mu"] - ref["mu"]) / np.abs(ref["mu"])) < 1e-13
    assert np.max(np.abs(res["std_dev"] - ref["std_dev"]) / ref["std_dev"]) < 1e-13
    assert np.array_equal(res["num_observed"], ref["num_observed"])
    # the edge cases: all-NaN rows for lengths 0 / 1, the noisy pixels are gone from all three matrices
    assert np.all(np.isnan(res["lya_1pzs"][-2:])) and np.all(np.isnan(y[-2:]))
    # the noisy-pixel rule: with it disabled, the grid points whose interpolated noise variance exceeds 1 are exactly
    # the ones the rule adds to the NaN pattern of lya_1pzs (which pixel masks leave alone)
    lya_loose, _, nv_loose = TS.training_matrices(sp["all_wavelengths"], sp["all_flux"], sp["all_noise_variance"],
                                                  sp["all_pixel_mask"], sp["z_qsos"], ref["rest_wavelengths"],
                                                  max_nv=np.inf)
    with np.errstate(invalid="ignore"):
        noisy = nv_loose > 1.0
    assert noisy.sum() >= 31 * 3                                          # every 97th spectrum has a noisy stretch
    assert np.array_equal(np.isnan(res["lya_1pzs"]), np.isnan(lya_loose) | noisy)
    assert np.all(np.isnan(y[noisy])) and np.all(np.isnan(res["rest_noise_variances"][noisy]))


@pytest.mark.gpu
def test_pairwise_covariance_matches_oracle(parity_case):
    from gp_dla_detection_b200 import api
    _, _, ref, res = parity_case
    X = ref["centered_rest_fluxes"]
    assert X.shape[0] % 32 and X.shape[0] % 64
    cov, counts = api.pairwise_covariance(X)
    assert np.array_equal(counts, ref["counts"])
    assert np.max(np.abs(cov - ref["cov"])) <= 1e-12 * np.abs(ref["cov"]).max()
    assert np.array_equal(cov, cov.T)
    cov2, counts2 = api.pairwise_covariance(X)
    assert np.array_equal(cov2, cov) and np.array_equal(counts2, counts)         # the same bits on every call


@pytest.mark.gpu
def test_pairwise_covariance_small_shapes_and_missing_pairs():
    from gp_dla_detection_b200 import api
    rng = np.random.default_rng(8)
    # N = 15 013 takes the largest number of row splits (8), whose partial tiles are summed in a fixed order
    for N, P in ((1, 1), (37, 65), (100, 130), (2049, 70), (15013, 70)):
        X = rng.standard_normal((N, P)) + 1.0
        X[rng.random(X.shape) < 0.2] = np.nan
        cov, counts = api.pairwise_covariance(X)
        C, n = TS.pairwise_covariance(X)
        assert np.array_equal(counts, n), (N, P)
        assert np.array_equal(np.isnan(cov), np.isnan(C)), (N, P)
        ok = ~np.isnan(C)
        if ok.any():
            assert np.max(np.abs(cov[ok] - C[ok])) <= 1e-12 * np.abs(C[ok]).max(), (N, P)
        cov2, counts2 = api.pairwise_covariance(X)
        assert np.array_equal(cov2, cov, equal_nan=True) and np.array_equal(counts2, counts), (N, P)
    X = rng.standard_normal((100, 70))
    X[50:, 3] = np.nan
    X[:50, 5] = np.nan                                                  # columns 3 and 5 are never observed together
    cov, counts = api.pairwise_covariance(X)
    assert counts[3, 5] == 0 and np.isnan(cov[3, 5]) and np.isnan(cov[5, 3])
    assert np.isfinite(np.delete(np.delete(cov, [3, 5], 0), [3, 5], 1)).all()


@pytest.mark.gpu
def test_disjoint_coverage_raises():
    """Every rest pixel is observed, but the two ends never in one spectrum: pca has no covariance there."""
    from gp_dla_detection_b200 import api
    rng = np.random.default_rng(9)
    sp = dict(all_wavelengths=[], all_flux=[], all_noise_variance=[], all_pixel_mask=[], z_qsos=np.full(8, 2.0))
    for q in range(8):
        x = np.arange(905.0, 1100.0, 0.3) if q < 4 else np.arange(1050.0, 1220.0, 0.3)
        sp["all_wavelengths"].append(3.0 * x)
        sp["all_flux"].append(1.0 + 0.1 * rng.standard_normal(x.size))
        sp["all_noise_variance"].append(np.full(x.size, 0.01))
        sp["all_pixel_mask"].append(np.zeros(x.size, dtype=bool))
    with pytest.raises(ValueError, match="pairwise covariance is undefined"):
        api.training_set(sp, 2)
    # a rest pixel observed fewer than twice: the host entry returns GPDLA_ERR_INVALID, the Python layer names it
    few = {k: v[:4] for k, v in sp.items() if k != "z_qsos"}
    few["z_qsos"] = sp["z_qsos"][:4]
    with pytest.raises(ValueError, match="is observed in 0 training spectra"):
        api.training_set(few, 2)


@pytest.mark.gpu
def test_initial_x_matches_oracle(parity_case):
    _, _, ref, res = parity_case
    k, P = 10, 1217
    top = ref["latent"][:k + 1]
    assert np.all(-np.diff(top) / top[1:] >= 1e-3), -np.diff(top) / top[1:]
    x, xr = res["initial_x"], ref["initial_x"]
    assert x.size == xr.size == P * (k + 1) + 3
    M, Mr = x[:P * k], xr[:P * k]
    assert np.max(np.abs(M - Mr)) <= 1e-9 * np.abs(Mr).max()
    assert np.max(np.abs(x[P * k:] - xr[P * k:]) / np.abs(xr[P * k:])) <= 1e-9


@pytest.mark.gpu
def test_device_chain_matches_host_entry():
    """Raw coadds -> preload_qsos_device -> training_set_device -> TrainingObjective on those CUDA tensors: the same
    objective and gradient bits as api.objective on the matrices of the host entry api.training_set."""
    import torch
    from gp_dla_detection_b200 import api
    rng = np.random.default_rng(12)
    raw, z = make_raw(48, 13, rng.uniform(3.0, 3.5, 48))
    pad = api._pad_raw(raw)
    t = {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in pad.items()}
    zt = torch.from_numpy(z).cuda()
    pre = api.preload_qsos_device(t["flux"], t["loglam"], t["ivar"], t["and_mask"], t["lengths"], zt)
    k = 10
    dev = api.training_set_device(pre["wavelengths"], pre["flux"], pre["noise_variance"], pre["pixel_mask"],
                                  pre["lengths"], zt, k)
    assert dev["centered_rest_fluxes"].is_cuda and isinstance(dev["initial_x"], np.ndarray)
    host_in = dict(wavelengths=pre["wavelengths"].cpu().numpy(), flux=pre["flux"].cpu().numpy(),
                   noise_variance=pre["noise_variance"].cpu().numpy(), pixel_mask=pre["pixel_mask"].cpu().numpy(),
                   lengths=pre["lengths"].cpu().numpy(), z_qsos=z)
    assert host_in["lengths"].min() > 0
    host = api.training_set(host_in, k)
    for n in ("lya_1pzs", "centered_rest_fluxes", "rest_noise_variances", "mu", "std_dev", "num_observed"):
        assert np.array_equal(dev[n].cpu().numpy(), host[n], equal_nan=True), n
    assert np.array_equal(dev["initial_x"], host["initial_x"])
    ev = api.TrainingObjective(dev["centered_rest_fluxes"], dev["lya_1pzs"], dev["rest_noise_variances"], k)
    assert ev.y.data_ptr() == dev["centered_rest_fluxes"].data_ptr()               # kept without a copy
    f, g = ev(dev["initial_x"])
    ev.close()
    fh, gh = api.objective(host["initial_x"], host["centered_rest_fluxes"], host["lya_1pzs"],
                           host["rest_noise_variances"])
    assert f == fh and np.array_equal(g, gh)
    assert np.isfinite(f) and np.all(np.isfinite(g))


@pytest.mark.gpu
def test_learn_qso_model_from_spectra_end_to_end():
    from gp_dla_detection_b200 import api, synthetic as syn
    _, sp = synthetic_training_spectra(2000, seed=31)
    k = 20
    learned = api.learn_qso_model_from_spectra(sp, k, max_iter=30)
    P = 1217
    assert learned["M"].shape == (P, k) and learned["mu"].shape == (P,) and learned["log_omega"].shape == (P,)
    assert learned["rest_wavelengths"].shape == (P,)
    for n in ("mu", "M", "log_omega"):
        assert np.all(np.isfinite(learned[n])), n
    assert all(np.isfinite(learned[n]) for n in ("log_c_0", "log_tau_0", "log_beta", "log_likelihood"))
    ts = api.training_set(sp, k)
    assert np.array_equal(ts["initial_x"], learned["initial_x"])
    f0, _ = api.objective(ts["initial_x"], ts["centered_rest_fluxes"], ts["lya_1pzs"], ts["rest_noise_variances"])
    assert learned["log_likelihood"] < f0
    samples, prior = syn.make_samples(2000), syn.make_prior(2000)
    spectra = syn.make_spectra(syn.make_model(k), 4, seed=5, dla_fraction=0.5)
    proc = api.DLAProcessor(learned, samples, prior)
    try:
        out = proc.process(spectra, return_sample_log_likelihoods=False)
    finally:
        proc.close()
    assert np.all(np.isfinite(out["p_dlas"]))
