"""CPU tests of the oracle itself (the checker must be pinned before it is trusted).

The reference ships no tests or fixtures (SURVEY.md section 4), so the anchors are: the reference's
own voigt.c compiled in oracle/_ref (and its committed outputs in tests/golden/voigt_reference.npz),
the literals printed in voigt.c, mpmath at 40 digits, and the dense multivariate normal."""
import math
import os

import numpy as np

from oracle import process_qsos_oracle as O
from oracle import ref as R
from conftest import boss_grid

ULP = np.finfo(np.float64).eps

# literals printed in the reference (voigt.c:151-184, :187-220): every entry
REF_LEADING = [
    1.34347262962625339e-07, 2.15386482180851912e-08, 7.48525170087141461e-09, 3.51375347286007472e-09,
    1.94112336271172934e-09, 1.18916112899713152e-09, 7.82448627128742997e-10, 5.42930932279390593e-10,
    3.92301197282493829e-10, 2.92796010451409027e-10, 2.24422239410389782e-10, 1.75895684469038289e-10,
    1.40338556137474778e-10, 1.13995374637743197e-10, 9.37706429662300083e-11, 7.79453203101192392e-11,
    6.55369055970184901e-11, 5.58100321584169051e-11, 4.77895916635794548e-11, 4.12301389852588843e-11,
    3.58872072638707592e-11, 3.12745536798214080e-11, 2.76337116167110415e-11, 2.44791750078032772e-11,
    2.15681362798480253e-11, 1.93850080479346101e-11, 1.72025364178111889e-11, 1.55051698336865945e-11,
    1.40504672409331934e-11, 1.28383057589411395e-11, 1.16264059622218997e-11]
REF_GAMMAS = [
    6.06075804241938613e+02, 1.54841462408931704e+02, 6.28964942715328164e+01, 3.17730561586147395e+01,
    1.82838676775503330e+01, 9.15463131005758157e+00, 6.08448802613156925e+00, 4.24977523573725779e+00,
    3.08542121666345803e+00, 2.31184525202557767e+00, 1.77687796208123139e+00, 1.39477990932179852e+00,
    1.11505539984541979e+00, 9.05885451682623022e-01, 7.45877170715450677e-01, 6.21261624902197052e-01,
    5.22994533400935269e-01, 4.44469874827484512e-01, 3.80923210837841919e-01, 3.28912390446060132e-01,
    2.85949711597237033e-01, 2.50280032040928802e-01, 2.20224061101442048e-01, 1.94686521675913549e-01,
    1.73082093051965591e-01, 1.54536566013816490e-01, 1.38539175663870029e-01, 1.24652675945279762e-01,
    1.12585442799479921e-01, 1.02045988802423507e-01, 9.27433783998286437e-02]


def test_tables_equal_reference_literals():
    assert np.array_equal(O.LEADING_CONSTANTS, np.array(REF_LEADING))
    assert np.array_equal(O.GAMMAS, np.array(REF_GAMMAS))
    assert O.INSTRUMENT_PROFILE.sum() == 1.0
    assert np.array_equal(O.INSTRUMENT_PROFILE, O.INSTRUMENT_PROFILE[::-1])


def test_voigt_matches_golden_reference_vectors(golden_dir):
    g = np.load(os.path.join(golden_dir, "voigt_reference.npz"))
    for i, (z, N, nl) in enumerate(g["cases"]):
        lam = g["lambdas"] if z < 3.5 else g["lambdas_hi"]
        a = O.voigt(lam, z, N, int(nl))
        assert a.shape == (lam.size - 6,)
        assert np.max(np.abs(a - g["profile_%d" % i])) <= 4 * ULP


def test_voigt_matches_compiled_reference(golden_dir):
    """Both restatements (Python and oracle/c) against the reference's own voigt.c: the profiles the compiled reference
    computed on the stored cases (tests/golden/voigt_reference.npz, written by tests/golden/make_golden.py), and, where
    oracle/_ref/voigt_ref.so has been built from the reference's source, 20 random profiles computed now."""
    g = np.load(os.path.join(golden_dir, "voigt_reference.npz"))
    for i, (z, N, nl) in enumerate(g["cases"]):
        lam = g["lambdas"] if z < 3.5 else g["lambdas_hi"]
        for voigt in (O.voigt, R.c_voigt):
            assert np.max(np.abs(voigt(lam, z, N, int(nl)) - g["profile_%d" % i])) <= 4 * ULP, (voigt.__name__, i)
    if not R.have_ref():
        return
    lam = boss_grid()
    rng = np.random.default_rng(0)
    for _ in range(20):
        z, logn, nl = rng.uniform(1.9, 2.9), rng.uniform(20, 23), int(rng.choice([1, 3, 5, 31]))
        assert np.max(np.abs(O.voigt(lam, z, 10 ** logn, nl) - R.ref_voigt(lam, z, 10 ** logn, nl))) <= 4 * ULP
    # the C restatement too
    assert np.max(np.abs(R.c_voigt(lam, 2.4, 1e21, 3) - R.ref_voigt(lam, 2.4, 1e21, 3))) <= 4 * ULP


def test_voigt_known_answers():
    lam = boss_grid(100)
    assert np.array_equal(O.voigt(lam, 2.2, 0.0, 3), np.ones(94))          # N = 0 -> no absorption, exactly
    a = O.voigt(boss_grid(), 2.3, 1e21, 3)
    assert a.min() >= 0.0 and a.max() <= 1.0
    centre = np.argmin(np.abs(boss_grid()[3:-3] - 1215.6701 * 3.3))
    assert a[centre] < 1e-20                                                # saturated core
    # more lines only ever absorb more
    assert np.all(O.voigt(boss_grid(), 2.3, 1e21, 31) <= O.voigt(boss_grid(), 2.3, 1e21, 3) + 4 * ULP)


def test_faddeeva_against_mpmath():
    import mpmath as mp
    from scipy.special import wofz
    mp.mp.dps = 40
    ys = O.GAMMAS[:3] / (math.sqrt(2) * O.SIGMA)
    xs = np.concatenate([np.linspace(0, 8, 33), np.geomspace(8, 8000, 40)])
    worst = 0.0
    for y in ys:
        for x in xs:
            z = mp.mpc(x, y)
            exact = (mp.exp(-z * z) * mp.erfc(-1j * z)).real
            worst = max(worst, abs(float(wofz(complex(x, y)).real / exact - 1)))
    assert worst < 5e-14


def test_log_mvnpdf_low_rank_against_dense():
    from scipy.stats import multivariate_normal
    rng = np.random.default_rng(1)
    for n, k in [(30, 3), (120, 20), (200, 7)]:
        M = rng.standard_normal((n, k)) * 0.3
        d = rng.uniform(0.05, 1.0, n)
        mu, y = rng.standard_normal(n), rng.standard_normal(n)
        dense = multivariate_normal.logpdf(y, mu, M @ M.T + np.diag(d))
        assert abs(O.log_mvnpdf_low_rank(y, mu, M, d) - dense) < 1e-9 * abs(dense)
        assert abs(R.c_log_mvnpdf_low_rank(y, mu, M, d) - dense) < 1e-9 * abs(dense)


def test_gemm_form_equals_literal_form(synthetic_inputs):
    """SURVEY.md 7.2: the Gram/projection reformulation the CUDA path uses equals the literal one."""
    si = synthetic_inputs
    sp = si["spectra"]
    rng = np.random.default_rng(2)
    n, k = 400, 20
    M = rng.standard_normal((n, k)) * 0.2
    mu, y = 1 + 0.1 * rng.standard_normal(n), 1 + 0.3 * rng.standard_normal(n)
    om2, v = rng.uniform(0.005, 0.02, n), rng.uniform(0.01, 0.2, n)
    a = np.clip(1 - np.exp(-np.linspace(-6, 6, n) ** 2), 0, 1)
    literal = O.log_mvnpdf_low_rank(y, mu * a, M * a[:, None], om2 * a ** 2 + v)
    d = a ** 2 * om2 + v
    w, u = a ** 2 / d, a * (y - a * mu) / d
    B = np.eye(k) + (M * w[:, None]).T @ M
    g = M.T @ u
    L = np.linalg.cholesky(B)
    zz = np.linalg.solve(L, g)
    gemm = -0.5 * (np.sum((y - a * mu) ** 2 / d) - zz @ zz + np.sum(np.log(d)) + 2 * np.sum(np.log(np.diag(L)))
                   + n * O.LOG_2PI)
    assert abs(gemm - literal) <= 1e-12 * abs(literal)


def test_c_engine_matches_numpy_engine(synthetic_inputs):
    si = synthetic_inputs
    sub = np.arange(0, 10000, 250)
    sp = {k: v[:2] for k, v in si["spectra"].items()}
    a = O.process_qsos(si["model"], si["samples"], sp, si["prior"], sample_subset=sub)
    b = O.process_qsos(si["model"], si["samples"], sp, si["prior"], sample_subset=sub, engine="c")
    rel = np.abs(a["sample_log_likelihoods_dla"] - b["sample_log_likelihoods_dla"]) / np.abs(a["sample_log_likelihoods_dla"])
    assert rel.max() < 1e-12
    assert np.array_equal(a["map_inds"], b["map_inds"])
    assert np.allclose(a["p_dlas"], b["p_dlas"], atol=1e-12)


def test_golden_process_qsos_regression(golden_dir):
    """The committed golden outputs are what the literal oracle produces (guards the fixtures)."""
    from test_gpu_parity import load_golden_problem
    model, samples, spectra, prior, expect = load_golden_problem(golden_dir)
    res = O.process_qsos(model, samples, spectra, prior)
    for k in ("log_likelihoods_no_dla", "log_likelihoods_dla", "sample_log_likelihoods_dla"):
        assert np.allclose(res[k], expect[k], rtol=1e-13, atol=0)
    assert np.array_equal(res["map_inds"], expect["map_inds"])


def test_lse_all_equal_and_masked_pixel_invariance(synthetic_inputs):
    si = synthetic_inputs
    sp = {k: v[:1] for k, v in si["spectra"].items()}
    sub = np.arange(0, 10000, 1000)
    base = O.process_qsos(si["model"], si["samples"], sp, si["prior"], sample_subset=sub, engine="c")
    # flagging an already unusable (out of window) pixel, or corrupting a masked pixel's flux, changes nothing
    sp2 = {k: ([x.copy() for x in v] if isinstance(v, list) else v.copy()) for k, v in sp.items()}
    masked = np.flatnonzero(sp2["all_pixel_mask"][0])
    sp2["all_flux"][0][masked] = 1e6
    sp2["all_pixel_mask"][0][0] = True
    again = O.process_qsos(si["model"], si["samples"], sp2, si["prior"], sample_subset=sub, engine="c")
    assert np.array_equal(base["sample_log_likelihoods_dla"], again["sample_log_likelihoods_dla"])
    # zero column density for every sample -> every sample likelihood equals the null likelihood
    s0 = dict(si["samples"]); s0["nhi_samples"] = np.zeros_like(s0["nhi_samples"])
    z = O.process_qsos(si["model"], s0, sp, si["prior"], sample_subset=sub, engine="c")
    assert np.allclose(z["sample_log_likelihoods_dla"], z["log_likelihoods_no_dla"][0], rtol=1e-13)
    assert abs(z["log_likelihoods_dla"][0] - z["log_likelihoods_no_dla"][0]) < 1e-10


def test_matlab_default_rng_stream():
    """rng('default') (multi-DLA resampling, ...meanflux.m:143) is MT19937 seed 5489."""
    r = np.random.RandomState(5489).rand(3)
    assert np.allclose(r, [0.8147236863931789, 0.9057919370756192, 0.1269868162935061], atol=1e-15)


def test_multi_oracle_engines_agree(synthetic_inputs):
    """Multi-DLA oracle: literal numpy loop vs the C engine, and the committed golden outputs."""
    from gp_dla_detection_b200 import synthetic as syn
    from oracle import process_qsos_multi_oracle as MO
    si = synthetic_inputs
    samples = syn.make_samples(10000, with_lls=True)
    sub = np.arange(11, 10000, 400)
    samples = {k: (v[sub] if isinstance(v, np.ndarray) else v) for k, v in samples.items()}
    sp = syn.make_spectra(si["model"], 1, seed=77, dla_fraction=1.0, meanflux=True, max_injected=2)
    kw = dict(Z_lls=samples["Z_lls"], Z_dla=samples["Z_dla"], max_dlas=3)
    a = MO.process_qsos_multi(si["model"], samples, sp, si["prior"], engine="numpy", **kw)
    b = MO.process_qsos_multi(si["model"], samples, sp, si["prior"], engine="c", **kw)
    assert np.array_equal(a["base_sample_inds"], b["base_sample_inds"])
    assert np.allclose(a["sample_log_likelihoods_dla"], b["sample_log_likelihoods_dla"], rtol=1e-12, equal_nan=True)
    assert np.allclose(a["model_posteriors"], b["model_posteriors"], atol=1e-12, equal_nan=True)
    assert abs(np.nansum(a["model_posteriors"]) - 1.0) < 1e-12
    # prior identity asserted by the reference (...meanflux.m:202)
    lp = np.exp(a["log_priors_dla"][0])
    lpno, lplls, _ = MO.multi_priors(si["prior"]["z_qsos"], si["prior"]["dla_ind"], float(sp["z_qsos"][0]), 3,
                                     samples["Z_lls"], samples["Z_dla"])
    frac = np.count_nonzero(si["prior"]["dla_ind"][si["prior"]["z_qsos"] < sp["z_qsos"][0] + O.prior_z_qso_increase]) / \
        np.count_nonzero(si["prior"]["z_qsos"] < sp["z_qsos"][0] + O.prior_z_qso_increase)
    assert abs(lp.sum() - frac) < 1e-4


def test_int8_digit_scheme_reproduces_fp64_gram():
    """The exact-product scheme of the INT8 tensor-core Gram path (signed 8-bit digits, truncated slice pairs, s32
    accumulators per diagonal) restated in integer NumPy: 6 digits are FP64-equivalent, 5 digits stay far inside
    the north-star tolerance, on a synthetic quasar and on one with 10 decades of noise variance and outliers;
    the s32 accumulators cannot overflow."""
    from oracle.int8_gram_oracle import fuzzed_and_plain
    plain, fuzz = fuzzed_and_plain(step=250, Ls=(5, 6))
    for res in (plain, fuzz):
        assert res[6][0] < 1e-12 and res[5][0] < 1e-10, res
        assert res[6][1] < 27 and res[5][1] < 27, res
