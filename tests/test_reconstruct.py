"""The fitted model of each quasar under chosen absorbers: the NumPy restatement against the dense Gaussian and the
existing oracles on the CPU; on the GPU the kernel against the restatement, its log-likelihood against the values the
fused hot-path kernels stored, calibration on spectra drawn from the model, and bit reproducibility."""
import ctypes
import math

import numpy as np
import pytest
from scipy.stats import multivariate_normal

from gp_dla_detection_b200 import _lib, api
from gp_dla_detection_b200 import params as P
from gp_dla_detection_b200 import synthetic as syn
from oracle import process_qsos_multi_oracle as MO
from oracle import process_qsos_oracle as O
from oracle import reconstruct_oracle as R

PLANE_RTOL = 1e-12     # planes: relative to each row's largest magnitude; scalars: relative
ABSORPTION_ATOL = 5e-15   # per absorber: the accuracy of one voigt profile (tests/test_gpu_parity.py), values in [0, 1]


# ------------------------------------------------------------------ inputs
def _spectra(model, Q, seed, meanflux=False, special=True):
    """Ragged synthetic spectra; with ``special`` also a heavily masked one, one whose window pixels are all masked
    and one with no pixel in the window."""
    sp = syn.make_spectra(model, Q, seed=seed, dla_fraction=0.3, meanflux=meanflux)
    if special:
        rng = np.random.default_rng(seed)
        lam, z = sp["all_wavelengths"][0], sp["z_qsos"][0]
        rest = lam / (1 + z)
        win = (rest >= P.DEFAULT.min_lambda) & (rest <= P.DEFAULT.max_lambda)
        heavy = sp["all_pixel_mask"][0] | (rng.random(lam.size) < 0.5)
        for w, f, v, m, zz in ((lam, sp["all_flux"][0], sp["all_noise_variance"][0], heavy, z),
                               (lam, sp["all_flux"][0], sp["all_noise_variance"][0], win | sp["all_pixel_mask"][0], z),
                               (lam[:5], sp["all_flux"][0][:5], sp["all_noise_variance"][0][:5],
                                np.zeros(5, bool), z)):
            sp["all_wavelengths"].append(w); sp["all_flux"].append(f); sp["all_noise_variance"].append(v)
            sp["all_pixel_mask"].append(m)
            sp["z_qsos"] = np.append(sp["z_qsos"], zz)
    return sp


def _absorbers(spectra, rng, A=4):
    """Up to A absorbers per quasar in its window: random ones, overlapping pairs and ones at the window edges."""
    Q = len(spectra["z_qsos"])
    z, n = np.full((Q, A), np.nan), np.full((Q, A), np.nan)
    for q in range(Q):
        lam, zq = spectra["all_wavelengths"][q], spectra["z_qsos"][q]
        rest = lam / (1 + zq)
        w = lam[(rest >= P.DEFAULT.min_lambda) & (rest <= P.DEFAULT.max_lambda)]
        if w.size == 0:
            continue
        lo, hi = w.min() / P.lya_wavelength - 1, w.max() / P.lya_wavelength - 1
        m = q % (A + 1)
        for b in range(m):
            kind = (q + b) % 4
            z[q, b] = lo if kind == 0 else hi if kind == 1 else rng.uniform(lo, hi)
            if kind == 3 and b > 0:
                z[q, b] = z[q, b - 1] + 1e-4                    # overlapping the previous one
            n[q, b] = 10.0 ** rng.uniform(19.5, 22.5)
    return z, n


def _processor(k=20, gram_digits=0, samples=None):
    return api.DLAProcessor(syn.make_model(k), samples or syn.make_samples(64), syn.make_prior(2000), device=0,
                            gram_digits=gram_digits)


# The three padded wavelengths on each side of the window are 10^(log10(lambda_end) -+ j pixel_spacing)
# (process_qsos.m:168-176), evaluated by the device's log10 / exp10 (the grid the fused kernels use) and by NumPy's in
# the oracle.  Each is within a few ulp of the exact value, but not bit-equal: log10(lambda_end) ~ 3.5 may differ by
# 3 ulp (1.3e-15 absolute, 3.1e-15 relative in the pad wavelength) and 10^x by 1.5 ulp (3.3e-16).  The three window
# pixels at each edge, whose 7-tap sums read the pads, are held to the oracle's own change under that shift.
PAD_RELATIVE = 4e-15


def _edge_tolerance(spectra, absorber_z, absorber_nhi, L_max):
    """[Q, L_max]: how far the oracle's absorption moves at the window's edge pixels when every pad wavelength moves by
    PAD_RELATIVE either way; zero elsewhere."""
    Q = len(spectra["z_qsos"])
    tol = np.zeros((Q, L_max))
    for q in range(Q):
        lam, zq = spectra["all_wavelengths"][q], spectra["z_qsos"][q]
        win = (lam / (1 + zq) >= P.DEFAULT.min_lambda) & (lam / (1 + zq) <= P.DEFAULT.max_lambda)
        absorbers = [(z, n) for z, n in zip(absorber_z[q], absorber_nhi[q]) if not np.isnan(z)]
        if not win.any() or not absorbers:
            continue
        pad = O.padded_wavelengths(lam[win])
        a = np.prod([O.voigt(pad, z, n, 3) for z, n in absorbers], axis=0)
        idx = np.flatnonzero(win)
        for sign in (1.0, -1.0):
            moved = pad.copy()
            moved[:3] *= 1.0 + sign * PAD_RELATIVE
            moved[-3:] *= 1.0 + sign * PAD_RELATIVE
            b = np.prod([O.voigt(moved, z, n, 3) for z, n in absorbers], axis=0)
            edge = np.r_[0:min(3, idx.size), max(idx.size - 3, 0):idx.size]
            tol[q, idx[edge]] = np.maximum(tol[q, idx[edge]], np.abs(b - a)[edge])
    return tol


def _assert_matches(got, ref, absorber_z=None, edge=None):
    """A product of m profiles is held to m times the accuracy of one, plus ``edge`` (see _edge_tolerance)."""
    m = np.ones(ref["absorption"].shape[0]) if absorber_z is None else \
        np.maximum(np.count_nonzero(~np.isnan(absorber_z), axis=1), 1)
    for nm in R.PLANES:
        g, r = got[nm], ref[nm]
        assert np.array_equal(np.isnan(g), np.isnan(r)), nm
        ok = ~np.isnan(r)
        if nm == "absorption":
            err = np.where(ok, np.abs(g - r), 0.0) - (0.0 if edge is None else edge)
            assert np.all(err <= ABSORPTION_ATOL * m[:, None]), (nm, (err / m[:, None]).max())
            continue
        scale = np.max(np.where(ok, np.abs(r), 0.0), axis=1, keepdims=True)
        err = np.where(ok, np.abs(g - r) / np.where(scale > 0, scale, 1.0), 0.0)
        assert np.all(err <= PLANE_RTOL), (nm, err.max())
    assert np.array_equal(got["num_pixels"], ref["num_pixels"])
    for nm in ("chi2", "log_likelihood"):
        g, r = got[nm], ref[nm]
        assert np.array_equal(np.isnan(g), np.isnan(r)), nm
        ok = ~np.isnan(r)
        assert np.all(np.abs(g[ok] - r[ok]) <= PLANE_RTOL * np.abs(r[ok])), (nm, np.max(np.abs(g[ok] - r[ok]) / np.abs(r[ok])))
    g, r = got["latent"], ref["latent"]
    assert np.array_equal(np.isnan(g), np.isnan(r))
    ok = ~np.isnan(r[:, 0])
    assert np.all(np.linalg.norm(g[ok] - r[ok], axis=1) <= PLANE_RTOL * np.linalg.norm(r[ok], axis=1))


# ------------------------------------------------------------------ CPU: the restatement
def test_woodbury_equals_dense_random():
    rng = np.random.default_rng(1)
    for n, k in ((30, 3), (80, 10), (200, 20), (300, 40)):
        aM = rng.standard_normal((n, k)) * rng.uniform(0.01, 0.5)
        d = rng.uniform(0.01, 0.3, n)
        r = rng.standard_normal(n) * 0.4
        _check_dense(aM, d, r)


def test_woodbury_equals_dense_synthetic_quasars():
    model = syn.make_model()
    sp = syn.make_spectra(model, 3, seed=4, dla_fraction=0.0)
    for q in range(3):
        lam, z = sp["all_wavelengths"][q], sp["z_qsos"][q]
        rest = lam / (1 + z)
        ind = (rest >= O.min_lambda) & (rest <= O.max_lambda) & ~sp["all_pixel_mask"][q]
        _, _, mu_t, M_t, om2_t = R.window_model(model, lam[ind], rest[ind], z, False)
        a = O.voigt(O.padded_wavelengths(lam[ind]), lam[ind].mean() / O.lya_wavelength - 1, 1e21, 3)
        _check_dense(M_t * a[:, None], om2_t * a ** 2 + sp["all_noise_variance"][q][ind],
                     sp["all_flux"][q][ind] - mu_t * a)


def _check_dense(aM, d, r):
    wb = R.woodbury(aM, d, r)
    K = aM @ aM.T + np.diag(d)
    Kinv_r = np.linalg.solve(K, r)
    Kinv_M = np.linalg.solve(K, aM)
    rel = lambda a, b: np.max(np.abs(a - b)) / np.max(np.abs(b))
    assert rel(wb["latent"], aM.T @ Kinv_r) < 1e-12
    assert abs(wb["chi2"] - r @ Kinv_r) < 1e-12 * abs(r @ Kinv_r)
    assert rel(wb["B_inv"], np.eye(aM.shape[1]) - aM.T @ Kinv_M) < 1e-12
    ref = multivariate_normal.logpdf(r, mean=np.zeros(r.size), cov=K)
    assert abs(wb["log_likelihood"] - ref) < 1e-12 * abs(ref)


def test_oracle_matches_process_qsos_oracle():
    """No absorber: the null log-likelihood; one sample's (z, N): that sample's log-likelihood."""
    model, samples = syn.make_model(), syn.make_samples(64)
    sp = syn.make_spectra(model, 3, seed=9, dla_fraction=0.5)
    for q in range(3):
        args = (sp["all_wavelengths"][q], sp["all_flux"][q], sp["all_noise_variance"][q], sp["all_pixel_mask"][q],
                float(sp["z_qsos"][q]))
        ref = O.process_one_quasar(model, samples, *args, sample_subset=np.array([5, 17]), engine="numpy")
        null = R.reconstruct_one(model, *args)
        assert abs(null["log_likelihood"] - ref["log_likelihoods_no_dla"]) <= 1e-12 * abs(ref["log_likelihoods_no_dla"])
        for i, s in enumerate((5, 17)):
            one = R.reconstruct_one(model, *args, [ref["sample_z_dlas"][i]], [samples["nhi_samples"][s]])
            want = ref["sample_log_likelihoods_dla"][i]
            assert abs(one["log_likelihood"] - want) <= 1e-12 * abs(want)


def test_oracle_matches_multi_oracle():
    """Mean-flux mode: the null model, a level-1 and a 2-absorber level-2 sample and the sub-DLA model of
    process_qsos_multi_oracle (its sample values carry -log S)."""
    model, samples = syn.make_model(), syn.make_samples(8, with_lls=True)
    sp = syn.make_spectra(model, 2, seed=11, dla_fraction=0.5, meanflux=True)
    S = 8
    base = np.array([np.roll(np.arange(S), 3), np.roll(np.arange(S), 5), np.roll(np.arange(S), 1)])
    for q in range(2):
        args = (sp["all_wavelengths"][q], sp["all_flux"][q], sp["all_noise_variance"][q], sp["all_pixel_mask"][q],
                float(sp["z_qsos"][q]))
        ref = MO.process_one_quasar_multi(model, samples, *args, max_dlas=2, base_sample_inds=base, engine="numpy")
        null = R.reconstruct_one(model, *args, meanflux=True)
        assert abs(null["log_likelihood"] - ref["log_likelihoods_no_dla"]) <= 1e-12 * abs(ref["log_likelihoods_no_dla"])
        zs = ref["min_z_dlas"] + (ref["max_z_dlas"] - ref["min_z_dlas"]) * samples["offset_samples"]
        nhi, lls = samples["nhi_samples"], samples["lls_nhi_samples"]
        for i in range(S):
            want = ref["sample_log_likelihoods_dla"][i, 0] + math.log(S)
            got = R.reconstruct_one(model, *args, [zs[i]], [nhi[i]], meanflux=True)["log_likelihood"]
            assert abs(got - want) <= 1e-12 * abs(want)
            want = ref["sample_log_likelihoods_lls"][i] + math.log(S)
            got = R.reconstruct_one(model, *args, [zs[i]], [lls[i]], meanflux=True)["log_likelihood"]
            assert abs(got - want) <= 1e-12 * abs(want)
            want = ref["sample_log_likelihoods_dla"][i, 1]
            if np.isnan(want):                  # the z-separation filter's
                continue
            p = base[0, i]
            got = R.reconstruct_one(model, *args, [zs[i], zs[p]], [nhi[i], nhi[p]], meanflux=True)["log_likelihood"]
            assert abs(got - (want + math.log(S))) <= 1e-12 * abs(want)


def _one(model, q=0, seed=2, **kw):
    sp = syn.make_spectra(model, 1, seed=seed, dla_fraction=0.0)
    return sp, R.reconstruct_one(model, sp["all_wavelengths"][q], sp["all_flux"][q], sp["all_noise_variance"][q],
                                 sp["all_pixel_mask"][q], float(sp["z_qsos"][q]), **kw)


def test_known_answer_zero_column_density():
    model = syn.make_model()
    sp, o = _one(model, absorber_z=[2.4], absorber_nhi=[0.0])
    a = o["absorption"][~np.isnan(o["absorption"])]
    assert a.size > 0 and np.all(a == 1.0)
    _, null = _one(model)
    for nm in R.PLANES:
        assert np.array_equal(o[nm], null[nm], equal_nan=True), nm


def test_known_answer_zero_M():
    model = dict(syn.make_model(), M=np.zeros((1217, 20)))
    _, o = _one(model, absorber_z=[2.4], absorber_nhi=[1e21])
    ok = ~np.isnan(o["continuum"])
    lam = _one(model)[0]["all_wavelengths"][0]
    z = _one(model)[0]["z_qsos"][0]
    mu = np.interp(lam / (1 + z), model["rest_wavelengths"], model["mu"])
    assert np.array_equal(o["continuum"][ok], mu[ok])
    assert np.all(o["continuum_sd"][ok] == 0.0)
    assert np.all(o["latent"] == 0.0)


def test_known_answer_masked_pixels_do_not_matter():
    model = syn.make_model()
    sp = syn.make_spectra(model, 1, seed=5, dla_fraction=0.0)
    mask = sp["all_pixel_mask"][0]
    assert mask.any()
    args = lambda f, v: (sp["all_wavelengths"][0], f, v, mask, float(sp["z_qsos"][0]), [2.5], [3e20])
    a = R.reconstruct_one(model, *args(sp["all_flux"][0], sp["all_noise_variance"][0]))
    f, v = sp["all_flux"][0].copy(), sp["all_noise_variance"][0].copy()
    f[mask] = 1e3
    v[mask] = 7.0
    b = R.reconstruct_one(model, *args(f, v))
    for nm in R.PLANES + ("latent", "chi2", "log_likelihood"):
        assert np.array_equal(a[nm], b[nm], equal_nan=True), nm


def test_map_absorbers_single_dla_results():
    samples = syn.make_samples(10)
    res = dict(min_z_dlas=np.array([2.0, 2.0, np.nan]), map_z_dlas=np.array([2.3, 2.1, np.nan]),
               map_inds=np.array([3, 7, -1]), p_dlas=np.array([0.9, 0.2, np.nan]),
               p_no_dlas=np.array([0.1, 0.8, np.nan]))
    z, n = api.map_absorbers(res, samples, 1)
    assert z.shape == (3, 1) and z[0, 0] == 2.3 and n[1, 0] == samples["nhi_samples"][7] and np.isnan(z[2, 0])
    z, n = api.map_absorbers(res, samples)
    assert z[0, 0] == 2.3 and np.all(np.isnan(z[1:]))
    z, n = api.map_absorbers(res, samples, "null")
    assert z.shape == (3, 0)
    with pytest.raises(ValueError):
        api.map_absorbers(res, samples, 2)
    with pytest.raises(ValueError):
        api.map_absorbers(res, samples, "sub_dla")


def test_map_absorbers_multi_results():
    samples = syn.make_samples(10, with_lls=True)
    mz = np.full((2, 2, 2), np.nan)
    mi = np.full((2, 2, 2), -1)
    mz[0, 0, 0], mi[0, 0, 0] = 2.2, 4
    mz[0, 1], mi[0, 1] = [2.2, 2.6], [4, 9]
    res = dict(min_z_dlas=np.array([2.0, 2.0]), max_z_dlas=np.array([3.0, 3.0]), MAP_z_dlas=mz, MAP_inds=mi,
               model_posteriors=np.array([[0.1, 0.1, 0.2, 0.6], [0.2, 0.7, 0.1, np.nan]]))
    z, n = api.map_absorbers(res, samples, 2)
    assert np.array_equal(z[0], [2.2, 2.6]) and np.array_equal(n[0], samples["nhi_samples"][[4, 9]])
    with pytest.raises(ValueError, match="sample_log_likelihoods_lls"):
        api.map_absorbers(res, samples, "sub_dla")
    ll = np.full((2, 10), -50.0)
    ll[1, 6] = -1.0
    res["sample_log_likelihoods_lls"] = ll
    z, n = api.map_absorbers(res, samples)
    assert z.shape == (2, 2) and np.array_equal(z[0], [2.2, 2.6])
    assert z[1, 0] == 2.0 + 1.0 * samples["offset_samples"][6] and n[1, 0] == samples["lls_nhi_samples"][6]
    assert np.isnan(z[1, 1])


# ------------------------------------------------------------------ GPU
@pytest.mark.gpu
@pytest.mark.parametrize("k", [10, 20, 40])
def test_kernel_matches_oracle(k):
    """About 200 quasars over k, meanflux and 0..4 absorbers (ragged, masked and empty ones included)."""
    proc = _processor(k)
    model = syn.make_model(k)
    try:
        for meanflux in (False, True):
            sp = _spectra(model, 31, seed=100 + k + meanflux, meanflux=meanflux)
            z, n = _absorbers(sp, np.random.default_rng(k))
            got = proc.reconstruct(sp, z, n, meanflux=meanflux)
            L_max = got["absorption"].shape[1]
            _assert_matches(got, R.reconstruct(model, sp, z, n, meanflux=meanflux, L_max=L_max), z,
                            _edge_tolerance(sp, z, n, L_max))
            assert np.count_nonzero(got["num_pixels"] == 0) == 2
        null = proc.reconstruct(sp, meanflux=True)
        _assert_matches(null, R.reconstruct(model, sp, meanflux=True, L_max=L_max))
    finally:
        proc.close()


@pytest.mark.gpu
def test_one_absorber_is_the_voigt_profile():
    proc = _processor()
    try:
        sp = _spectra(syn.make_model(), 4, seed=3, special=False)
        z, n = _absorbers(sp, np.random.default_rng(0), A=1)
        z[:, 0], n[:, 0] = 2.4, 2e21
        got = proc.reconstruct(sp, z, n)
        for q in range(4):
            lam, zq = sp["all_wavelengths"][q], sp["z_qsos"][q]
            rest = lam / (1 + zq)
            win = (rest >= P.DEFAULT.min_lambda) & (rest <= P.DEFAULT.max_lambda)
            ref = api.voigt(O.padded_wavelengths(lam[win]), 2.4, 2e21, 3)
            # bit-equal away from the pads, whose wavelengths NumPy rounds differently (see _edge_tolerance)
            assert np.array_equal(got["absorption"][q, :lam.size][win][3:-3], ref[3:-3])
            edge = _edge_tolerance(sp, z[:, :1], n[:, :1], got["absorption"].shape[1])[q, :lam.size][win]
            assert np.all(np.abs(got["absorption"][q, :lam.size][win] - ref) <= edge + ABSORPTION_ATOL)
        z[:, 0], n[:, 0] = 2.4, 0.0
        a = proc.reconstruct(sp, z, n)["absorption"]
        assert np.all(a[~np.isnan(a)] == 1.0)
    finally:
        proc.close()


def _planes(spectra):
    import torch
    pad = api.pad_spectra(spectra)
    up = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dtype=dt)).cuda()
    return (up(pad["wavelengths"], np.float64), up(pad["flux"], np.float64), up(pad["noise_variance"], np.float64),
            up(pad["pixel_mask"], np.uint8), up(pad["lengths"], np.int32), up(pad["z_qsos"], np.float64))


def _close(a, b, rtol=1e-10):
    ok = ~np.isnan(b)
    assert np.array_equal(np.isnan(a), np.isnan(b))
    err = np.abs(a[ok] - b[ok]) / np.abs(b[ok])
    assert np.all(err <= rtol), err.max()


@pytest.mark.gpu
@pytest.mark.parametrize("gram_digits", [0, -1])
def test_single_dla_hot_path_log_likelihoods(gram_digits):
    samples = syn.make_samples(2000)
    model = syn.make_model()
    proc = api.DLAProcessor(model, samples, syn.make_prior(), device=0, gram_digits=gram_digits)
    try:
        sp = syn.make_spectra(model, 40, seed=21, dla_fraction=0.5)
        planes = _planes(sp)
        out = proc.process_device(*planes, return_sample_log_likelihoods=True)
        host = {k: v.cpu().numpy() for k, v in out.items()}
        Q = host["map_inds"].size
        z, n = api.map_absorbers(out, samples, 1)
        rec = proc.reconstruct_device(*planes, absorber_z=z, absorber_nhi=n)
        _close(rec["log_likelihood"].cpu().numpy(), host["sample_log_likelihoods_dla"][np.arange(Q), host["map_inds"]])
        z, n = api.map_absorbers(out, samples, "null")
        _close(proc.reconstruct_device(*planes, absorber_z=z, absorber_nhi=n)["log_likelihood"].cpu().numpy(),
               host["log_likelihoods_no_dla"])
        rng = np.random.default_rng(gram_digits + 7)
        for _ in range(10):
            i = rng.integers(0, samples["offset_samples"].size, Q)
            zi = host["min_z_dlas"] + (host["max_z_dlas"] - host["min_z_dlas"]) * samples["offset_samples"][i]
            rec = proc.reconstruct_device(*planes, absorber_z=zi[:, None], absorber_nhi=samples["nhi_samples"][i][:, None])
            _close(rec["log_likelihood"].cpu().numpy(), host["sample_log_likelihoods_dla"][np.arange(Q), i])
    finally:
        proc.close()


@pytest.mark.gpu
@pytest.mark.parametrize("gram_digits", [0, -1])
def test_multi_dla_hot_path_log_likelihoods(gram_digits):
    samples = syn.make_samples(2000, with_lls=True)
    model = syn.make_model()
    S = samples["offset_samples"].size
    proc = api.DLAProcessor(model, samples, syn.make_prior(), device=0, gram_digits=gram_digits)
    try:
        sp = syn.make_spectra(model, 40, seed=23, dla_fraction=0.5, meanflux=True, second_dla_fraction=0.5)
        planes = _planes(sp)
        out = proc.process_multi_device(*planes, max_dlas=4, return_samples=True)
        host = {k: v.cpu().numpy() for k, v in out.items()}
        Q = host["min_z_dlas"].size
        reached = 0
        for j in range(1, 5):
            z, n = api.map_absorbers(out, samples, j)
            ll = proc.reconstruct_device(*planes, absorber_z=z, absorber_nhi=n, meanflux=True)["log_likelihood"]
            ind = host["MAP_inds"][:, j - 1, 0]
            ok = ind >= 0
            reached += np.count_nonzero(ok)
            want = host["sample_log_likelihoods_dla"][np.arange(Q), j - 1, np.maximum(ind, 0)] + math.log(S)
            _close(ll.cpu().numpy()[ok], want[ok])
        assert reached > Q
        z, n = api.map_absorbers(out, samples, "sub_dla")
        ll = proc.reconstruct_device(*planes, absorber_z=z, absorber_nhi=n, meanflux=True)["log_likelihood"].cpu().numpy()
        lls = host["sample_log_likelihoods_lls"]
        ok = ~np.all(np.isnan(lls), axis=1)
        _close(ll[ok], np.nanmax(lls[ok], axis=1) + math.log(S))
        z, n = api.map_absorbers(out, samples)               # the most probable model runs
        assert z.shape == (Q, 4)
        proc.reconstruct_device(*planes, absorber_z=z, absorber_nhi=n, meanflux=True)
    finally:
        proc.close()


def _draw_calibration(model, Q, rng):
    """Spectra drawn from the (single-DLA) model with their latent x: window pixels of the BOSS grid, 2 % masked, a
    quarter with one absorber applied with the oracle's convolved profile."""
    k = model["M"].shape[1]
    sp = dict(all_wavelengths=[], all_flux=[], all_noise_variance=[], all_pixel_mask=[], z_qsos=[])
    x_true, truth, az, an = np.empty((Q, k)), [], np.full((Q, 1), np.nan), np.full((Q, 1), np.nan)
    for q in range(Q):
        z = 2.2 + rng.gamma(2.0, 0.3)
        j0 = math.ceil((math.log10(P.DEFAULT.min_lambda * (1 + z)) - 3.5563) / 1e-4)
        j1 = math.floor((math.log10(P.DEFAULT.max_lambda * (1 + z)) - 3.5563) / 1e-4)
        lam = 10.0 ** (3.5563 + 1e-4 * np.arange(j0, j1 + 1))
        rest = lam / (1 + z)
        keep = (rest >= P.DEFAULT.min_lambda) & (rest <= P.DEFAULT.max_lambda)
        lam, rest = lam[keep], rest[keep]
        mu, M, _, _, om2 = R.window_model(model, lam, rest, z, False)
        x = rng.standard_normal(k)
        a = np.ones(lam.size)
        if q % 4 == 0:
            az[q, 0] = rng.uniform(lam.min() / P.lya_wavelength - 1, lam.max() / P.lya_wavelength - 1)
            an[q, 0] = 10.0 ** rng.uniform(20.0, 21.5)
            a = O.voigt(O.padded_wavelengths(lam), az[q, 0], an[q, 0], 3)
        v = (0.1 + 0.4 * rng.random(lam.size)) ** 2
        flux = a * (mu + M @ x + np.sqrt(om2) * rng.standard_normal(lam.size)) + np.sqrt(v) * rng.standard_normal(lam.size)
        for key, val in (("all_wavelengths", lam), ("all_flux", flux), ("all_noise_variance", v),
                         ("all_pixel_mask", rng.random(lam.size) < 0.02), ("z_qsos", z)):
            sp[key].append(val)
        x_true[q] = x
        truth.append(mu + M @ x)
    sp["z_qsos"] = np.asarray(sp["z_qsos"])
    return sp, x_true, truth, az, an


@pytest.mark.gpu
def test_calibration_on_spectra_drawn_from_the_model():
    model = syn.make_model()
    k, Q = 20, 2000
    sp, x_true, truth, az, an = _draw_calibration(model, Q, np.random.default_rng(77))
    proc = _processor(k)
    try:
        got = proc.reconstruct(sp, az, an)
    finally:
        proc.close()
    quad, num, den = 0.0, 0.0, 0
    for q in range(Q):
        o = R.reconstruct_one(model, sp["all_wavelengths"][q], sp["all_flux"][q], sp["all_noise_variance"][q],
                              sp["all_pixel_mask"][q], float(sp["z_qsos"][q]), az[q], an[q])
        e = got["latent"][q] - x_true[q]
        quad += e @ o["B"] @ e
        L = len(sp["all_wavelengths"][q])
        used = ~sp["all_pixel_mask"][q]
        t = (got["continuum"][q, :L] - truth[q]) / got["continuum_sd"][q, :L]
        num += np.sum(t[used] ** 2)
        den += np.count_nonzero(used)
    assert abs(quad / (Q * k) - 1.0) < 0.04, quad / (Q * k)
    assert abs(num / den - 1.0) < 0.15, num / den


@pytest.mark.gpu
def test_bits_repeat_host_device_and_fresh_meanflux_context():
    model = syn.make_model()
    sp = _spectra(model, 20, seed=31, meanflux=True)
    z, n = _absorbers(sp, np.random.default_rng(3))
    fresh = _processor()                       # no process_multi call before: forest constants come with the context
    try:
        a = fresh.reconstruct(sp, z, n, meanflux=True)
        b = fresh.reconstruct(sp, z, n, meanflux=True)
        dev = fresh.reconstruct_device(*_planes(sp), absorber_z=z, absorber_nhi=n, meanflux=True)
        for nm in a:
            assert np.array_equal(a[nm], b[nm], equal_nan=True), nm
            assert np.array_equal(a[nm], dev[nm].cpu().numpy(), equal_nan=True), nm
        L_max = a["absorption"].shape[1]
        _assert_matches(a, R.reconstruct(model, sp, z, n, meanflux=True, L_max=L_max), z, _edge_tolerance(sp, z, n, L_max))
    finally:
        fresh.close()


@pytest.mark.gpu
def test_argument_checks():
    lib = _lib.load()
    proc = _processor()
    sp = _spectra(syn.make_model(), 2, seed=1, special=False)
    try:
        with pytest.raises(ValueError):
            proc.reconstruct(sp, np.zeros((4, 5)), np.zeros((4, 5)))
        for bad_z, bad_n in ((-1.0, 1e20), (2.3, -1.0), (2.3, np.inf), (np.inf, 1e20)):
            with pytest.raises(_lib.GpdlaError) as e:
                proc.reconstruct(sp, np.full((2, 1), bad_z), np.full((2, 1), bad_n))
            assert e.value.code == _lib.GPDLA_ERR_INVALID
        pad = api.pad_spectra(sp)
        vp = lambda a: ctypes.c_void_p(np.ascontiguousarray(a).ctypes.data)
        arrs = [np.ascontiguousarray(pad[k]) for k in ("wavelengths", "flux", "noise_variance")]
        mk, ln, zq = (np.ascontiguousarray(pad["pixel_mask"], dtype=np.uint8),
                      np.ascontiguousarray(pad["lengths"], dtype=np.int32), np.ascontiguousarray(pad["z_qsos"]))
        res = _lib.GpdlaReconstruction()
        call = lambda ctx, mf, A: lib.gpdla_reconstruct(ctx, 2, arrs[0].shape[1], *[vp(a) for a in arrs], vp(mk), vp(ln),
                                                        vp(zq), mf, A, None, None, ctypes.byref(res))
        assert call(proc._ctx, 2, 0) == _lib.GPDLA_ERR_INVALID
        assert call(proc._ctx, 0, 1) == _lib.GPDLA_ERR_INVALID        # absorber arrays NULL with num_absorbers > 0
        empty = ctypes.c_void_p()
        _lib.check(lib.gpdla_create(ctypes.byref(empty), 0))
        try:
            assert call(empty, 0, 0) == _lib.GPDLA_ERR_STATE
        finally:
            lib.gpdla_destroy(empty)
    finally:
        proc.close()
