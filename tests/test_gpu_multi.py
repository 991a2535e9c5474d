"""GPU parity tests of the multi-DLA + sub-DLA + mean-flux path
(multi_dlas/process_qsos_multiple_dlas_meanflux.m) through the C ABI, against the oracle."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
LL_RTOL = 1e-10     # implementation bar (north_star: 1e-8)
P_ATOL = 1e-6


def load_golden_multi(golden_dir):
    g = np.load(os.path.join(golden_dir, "process_qsos_multi_small.npz"))
    b = np.load(os.path.join(golden_dir, "process_qsos_small.npz"))
    model = dict(rest_wavelengths=b["model_rest_wavelengths"], mu=b["model_mu"], M=b["model_M"],
                 log_omega=b["model_log_omega"], log_c_0=b["model_scalars"][0], log_tau_0=b["model_scalars"][1],
                 log_beta=b["model_scalars"][2])
    samples = {k: g[k] for k in ("offset_samples", "log_nhi_samples", "nhi_samples", "lls_nhi_samples")}
    samples["Z_lls"], samples["Z_dla"] = float(g["Z"][0]), float(g["Z"][1])
    prior = dict(z_qsos=b["prior_z_qsos"], dla_ind=b["prior_dla_ind"])
    spectra = {k: [g["%s_%d" % (k, q)] for q in range(2)]
               for k in ("all_wavelengths", "all_flux", "all_noise_variance", "all_pixel_mask")}
    spectra["z_qsos"] = g["z_qsos"]
    expect = {k[4:]: g[k] for k in g.files if k.startswith("out_")}
    return model, samples, spectra, prior, expect


def assert_multi_parity(res, ref, check_base=True, ll_rtol=LL_RTOL, check_map=True):
    """``ll_rtol``: the log-likelihood bar (1e-9 for the 5-digit INT8 Gram and for extreme inputs, as on the
    single-DLA path); ``check_map=False`` leaves the MAP to a caller that checks it only where it is tie-free."""
    if check_base:
        assert np.array_equal(res["base_sample_inds"], ref["base_sample_inds"])
    a, b = res["sample_log_likelihoods_dla"], ref["sample_log_likelihoods_dla"]
    assert np.array_equal(np.isnan(a), np.isnan(b))                      # z-separation filter / early exit pattern
    assert np.allclose(a, b, rtol=ll_rtol, atol=0, equal_nan=True)
    assert np.array_equal(np.isnan(res["sample_log_likelihoods_lls"]), np.isnan(ref["sample_log_likelihoods_lls"]))
    assert np.allclose(res["sample_log_likelihoods_lls"], ref["sample_log_likelihoods_lls"], rtol=ll_rtol, atol=0,
                       equal_nan=True)
    for k in ("log_likelihoods_no_dla", "log_likelihoods_lls", "log_likelihoods_dla", "log_posteriors_no_dla",
              "log_posteriors_lls", "log_posteriors_dla"):
        assert np.allclose(res[k], ref[k], rtol=ll_rtol, atol=0, equal_nan=True), k
    for k in ("log_priors_no_dla", "log_priors_lls", "log_priors_dla", "min_z_dlas", "max_z_dlas"):
        assert np.allclose(res[k], ref[k], rtol=1e-13, atol=0, equal_nan=True), k
    # MAP: same arg-max sample, except for exact ties -- at levels >= 2 resampling with replacement produces
    # samples that describe the same set of DLAs in a different order, whose likelihoods agree to rounding
    Q, MD = res["MAP_inds"].shape[:2]
    for q in range(Q if check_map else 0):
        for l in range(MD):
            i, j = res["MAP_inds"][q, l, 0], ref["MAP_inds"][q, l, 0]
            if i == j:
                assert np.array_equal(res["MAP_inds"][q, l], ref["MAP_inds"][q, l])
                assert np.allclose(res["MAP_z_dlas"][q, l], ref["MAP_z_dlas"][q, l], rtol=1e-13, atol=0, equal_nan=True)
                assert np.allclose(res["MAP_log_nhis"][q, l], ref["MAP_log_nhis"][q, l], rtol=1e-13, atol=0, equal_nan=True)
            else:
                assert l >= 1 and i >= 0 and j >= 0
                assert abs(b[q, i, l] - b[q, j, l]) <= 1e-11 * abs(b[q, j, l]), (q, l, i, j)
                assert np.allclose(np.sort(res["MAP_z_dlas"][q, l, :l + 1]), np.sort(ref["MAP_z_dlas"][q, l, :l + 1]),
                                   rtol=1e-13, atol=0)
    for k in ("model_posteriors", "p_no_dlas", "p_lls", "p_dlas"):
        assert np.allclose(res[k], ref[k], rtol=0, atol=P_ATOL, equal_nan=True), k


@pytest.fixture(scope="module")
def api():
    from gp_dla_detection_b200 import api as A
    return A


def test_matlab_default_rand_stream(api):
    assert np.array_equal(api.matlab_default_rand(1000), np.random.RandomState(5489).random_sample(1000))


def test_multi_golden_small(api, golden_dir):
    model, samples, spectra, prior, expect = load_golden_multi(golden_dir)
    res = api.process_qsos_multiple_dlas_meanflux(model, samples, spectra, prior, max_dlas=3)
    assert_multi_parity(res, expect)


def test_multi_against_oracle(api, synthetic_inputs):
    """2000 samples, 4 levels, spectra with up to two injected DLAs; the resampling must reproduce the
    oracle's base_sample_inds (MATLAB rng('default') + randsample) and every level's likelihoods."""
    from gp_dla_detection_b200 import synthetic as syn
    from oracle import process_qsos_multi_oracle as MO
    si = synthetic_inputs
    samples = syn.make_samples(2000, with_lls=True)
    sp = syn.make_spectra(si["model"], 3, seed=5, dla_fraction=0.7, meanflux=True, max_injected=2)
    ref = MO.process_qsos_multi(si["model"], samples, sp, si["prior"], Z_lls=samples["Z_lls"], Z_dla=samples["Z_dla"])
    res = api.process_qsos_multiple_dlas_meanflux(si["model"], samples, sp, si["prior"])
    same = np.mean(res["base_sample_inds"] == ref["base_sample_inds"])
    assert same > 0.999, same            # a draw within ~1e-13 of a CDF edge may legitimately differ
    # with the oracle's indices given, everything must agree to rounding
    res2 = api.process_qsos_multiple_dlas_meanflux(si["model"], samples, sp, si["prior"],
                                                   base_sample_inds=ref["base_sample_inds"])
    assert_multi_parity(res2, ref)
    # the two-DLA quasars are found as such
    assert np.array_equal(np.argmax(res["model_posteriors"], axis=1), np.argmax(ref["model_posteriors"], axis=1))


def test_multi_rank_40(api, synthetic_inputs):
    """The level loop at k = 40: MODE 1 / MODE 2 of the INT8 producing kernel with its contract-only passes, against
    the oracle with the oracle's resampling indices, and against the FP64 DMMA path."""
    from gp_dla_detection_b200 import synthetic as syn
    from oracle import process_qsos_multi_oracle as MO
    si = synthetic_inputs
    m40 = syn.make_model(40)
    samples = syn.make_samples(700, with_lls=True)
    sp = syn.make_spectra(m40, 2, seed=6, dla_fraction=1.0, meanflux=True, max_injected=2)
    ref = MO.process_qsos_multi(m40, samples, sp, si["prior"], Z_lls=samples["Z_lls"], Z_dla=samples["Z_dla"], max_dlas=3)
    for digits in (6, -1):
        res = api.process_qsos_multiple_dlas_meanflux(m40, samples, sp, si["prior"], max_dlas=3, gram_digits=digits,
                                                      base_sample_inds=ref["base_sample_inds"])
        assert_multi_parity(res, ref)


def test_multi_empty_and_batched(api, synthetic_inputs):
    from gp_dla_detection_b200 import synthetic as syn
    si = synthetic_inputs
    samples = syn.make_samples(500, with_lls=True)
    sp = syn.make_spectra(si["model"], 5, seed=8, dla_fraction=0.5, meanflux=True)
    sp["all_pixel_mask"][2][:] = True
    one = api.process_qsos_multiple_dlas_meanflux(si["model"], samples, sp, si["prior"], max_dlas=2)
    two = api.process_qsos_multiple_dlas_meanflux(si["model"], samples, sp, si["prior"], max_dlas=2, batch_quasars=2)
    for k in one:
        assert np.array_equal(one[k], two[k], equal_nan=True), k
    assert np.isnan(one["log_likelihoods_no_dla"][2]) and np.all(np.isnan(one["log_likelihoods_dla"][2]))
    assert np.all(np.isnan(one["model_posteriors"][2])) and np.all(one["MAP_inds"][2] == -1)
    assert not np.isnan(one["log_priors_no_dla"][2])            # priors are set before the skip (...meanflux.m:204-216)
    assert np.all(np.isfinite(one["log_likelihoods_dla"][[0, 1, 3, 4]]))
