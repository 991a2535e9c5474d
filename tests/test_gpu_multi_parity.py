"""The multi-DLA path (multi_dlas/process_qsos_multiple_dlas_meanflux.m) held to the single-DLA path's parity bar:
split batches, the FP64 fallback list, every rank, Gram arithmetic and line count, tile edges, sample order, early exit,
prior edges, extreme spectra and every entry, against the oracle.

The kernels are compared with the oracle under given ``base_sample_inds`` taken from the oracle's own run, so that
parity does not depend on draws within ~1e-13 of a CDF edge.  The unmarked tests pin the oracle behaviour the GPU
tests rely on."""
import math

import numpy as np
import pytest

from test_gpu_multi import LL_RTOL, assert_multi_parity

gpu = pytest.mark.gpu
LEVEL_RTOL = 1e-13      # level evidences summed in another sample order


@pytest.fixture(scope="module")
def api():
    from gp_dla_detection_b200 import api as A
    return A


def _oracle(model, samples, spectra, prior, **kw):
    from oracle import process_qsos_multi_oracle as MO
    return MO.process_qsos_multi(model, samples, spectra, prior, Z_lls=samples["Z_lls"], Z_dla=samples["Z_dla"], **kw)


def _quasars(spectra, rows):
    return {k: ([v[i] for i in rows] if isinstance(v, list) else np.asarray(v)[rows]) for k, v in spectra.items()}


def _rows(res, rows):
    return {k: np.asarray(v)[rows] for k, v in res.items()}


def assert_same(a, b, rows=None):
    """Every output bit for bit (NaN where NaN), optionally on a subset of quasars."""
    assert a.keys() == b.keys()
    for k in a:
        x, y = np.asarray(a[k]), np.asarray(b[k])
        if rows is not None:
            x, y = x[rows], y[rows]
        assert x.dtype == y.dtype and np.array_equal(x, y, equal_nan=True), k


def _zero_noise(spectra, q, picks):
    """noise_variance = 0 on used pixels redward of every sampled DLA (max_z_dla stops 43 pixels short of the
    quasar's Lyman alpha): the absorption never reaches zero there, so d = a^2 omega^2 stays positive."""
    w = np.asarray(spectra["all_wavelengths"][q]) / (1 + spectra["z_qsos"][q])
    used = np.flatnonzero(~np.asarray(spectra["all_pixel_mask"][q]) & (w >= 911.75) & (w <= 1215.75))
    spectra["all_noise_variance"][q][used[picks]] = 0.0


def _force_early_exit(model, samples, spectra, prior, ref, rows, **kw):
    """Each level-2 sample of ``rows`` is its own partner: the separation filter removes them all and the level loop
    stops after level 2.  Returns the given indices and the oracle's results under them."""
    S = len(samples["offset_samples"])
    base = ref["base_sample_inds"].copy()
    base[rows, :, 0] = np.arange(S)
    forced = _oracle(model, samples, _quasars(spectra, rows), prior, base_sample_inds=base[rows], **kw)
    out = {k: v.copy() for k, v in ref.items()}
    for k in out:
        out[k][rows] = forced[k]
    return base, out


def _assert_stopped_after_level_1(res, q):
    ll = res["log_likelihoods_dla"][q]
    assert np.isfinite(ll[0]) and np.all(np.isnan(ll[1:]))
    assert np.all(np.isnan(res["sample_log_likelihoods_dla"][q][:, 1:]))
    assert np.all(res["MAP_inds"][q, 1:] == -1) and np.isnan(res["p_dlas"][q])


# ------------------------------------------------------------------------------------------------ the oracle (CPU)
def test_oracle_sample_permutation_with_mapped_partners(synthetic_inputs):
    """Permuting every per-sample array and mapping the partners through the permutation permutes the sample
    log-likelihoods bit for bit, maps the MAP through the permutation and leaves the level evidences unchanged."""
    from gp_dla_detection_b200 import synthetic as syn
    si = synthetic_inputs
    S = 33
    samples = syn.make_samples(S, with_lls=True)
    sp = syn.make_spectra(si["model"], 1, seed=201, dla_fraction=1.0, meanflux=True, second_dla_fraction=1.0)
    a = _oracle(si["model"], samples, sp, si["prior"])
    perm = np.random.default_rng(3).permutation(S)
    sperm = {k: (v[perm] if np.ndim(v) else v) for k, v in samples.items()}
    base = np.argsort(perm)[a["base_sample_inds"][:, perm, :]]
    b = _oracle(si["model"], sperm, sp, si["prior"], base_sample_inds=base)
    assert np.array_equal(a["sample_log_likelihoods_dla"][:, perm, :], b["sample_log_likelihoods_dla"], equal_nan=True)
    assert np.array_equal(a["sample_log_likelihoods_lls"][:, perm], b["sample_log_likelihoods_lls"])
    ok = b["MAP_inds"] >= 0
    assert np.array_equal(ok, a["MAP_inds"] >= 0) and np.array_equal(perm[b["MAP_inds"][ok]], a["MAP_inds"][ok])
    assert np.allclose(a["log_likelihoods_dla"], b["log_likelihoods_dla"], rtol=LEVEL_RTOL, atol=0, equal_nan=True)
    assert np.isfinite(a["log_likelihoods_dla"][0, 1])                      # the permutation reached level 2


def test_oracle_forced_early_exit(synthetic_inputs):
    from gp_dla_detection_b200 import synthetic as syn
    si = synthetic_inputs
    samples = syn.make_samples(24, with_lls=True)
    sp = syn.make_spectra(si["model"], 2, seed=202, dla_fraction=0.5, meanflux=True)
    ref = _oracle(si["model"], samples, sp, si["prior"])
    assert np.all(np.isfinite(ref["log_likelihoods_dla"][:, :2]))
    _, forced = _force_early_exit(si["model"], samples, sp, si["prior"], ref, [1])
    _assert_stopped_after_level_1(forced, 1)
    assert np.all(np.isnan(forced["model_posteriors"][1]))                  # NaN levels propagate through the sum
    assert np.array_equal(forced["base_sample_inds"][1, :, 0], np.arange(24))
    assert np.all(forced["base_sample_inds"][1, :, 1:] == 0)                # levels never reached keep their zeros
    assert_same(_rows(forced, [0]), _rows(ref, [0]))


def _edge_priors(prior):
    n = len(prior["z_qsos"])
    return dict(no_dlas=dict(z_qsos=prior["z_qsos"], dla_ind=np.zeros(n, dtype=bool)),
                all_dlas=dict(z_qsos=prior["z_qsos"], dla_ind=np.ones(n, dtype=bool)),
                catalogue=prior)


def test_oracle_prior_edges(synthetic_inputs):
    """multi_priors at the edges, against hand values: a catalogue without DLAs (-inf), one where every quasar is
    a DLA (log of a negative count for the null model), a quasar below every catalogue quasar (0 / 0)."""
    from oracle import process_qsos_multi_oracle as MO
    prior = synthetic_inputs["prior"]
    Z_lls, Z_dla = 0.18, 0.82
    pr = _edge_priors(prior)
    z = 2.5
    no, lls, dla = MO.multi_priors(pr["no_dlas"]["z_qsos"], pr["no_dlas"]["dla_ind"], z, 4, Z_lls, Z_dla)
    assert no == 0.0 and lls == -np.inf and np.all(dla == -np.inf)
    no, lls, dla = MO.multi_priors(pr["all_dlas"]["z_qsos"], pr["all_dlas"]["dla_ind"], z, 4, Z_lls, Z_dla)
    assert np.isnan(no) and lls == math.log(Z_lls) - math.log(Z_dla)
    assert np.all(dla[:3] == -np.inf) and dla[3] == 0.0
    no, lls, dla = MO.multi_priors(prior["z_qsos"], prior["dla_ind"], z, 2, Z_lls, Z_dla)
    n = np.count_nonzero(prior["z_qsos"] < z + MO.O.prior_z_qso_increase)
    d = np.count_nonzero(prior["dla_ind"][prior["z_qsos"] < z + MO.O.prior_z_qso_increase])
    assert np.allclose(dla, np.log([d / n - (d / n) ** 2, (d / n) ** 2]), rtol=1e-14, atol=0)
    assert np.isclose(no, math.log((n - d - Z_lls * d / Z_dla) / n), rtol=1e-14, atol=0)
    z_low = float(np.min(prior["z_qsos"])) - MO.O.prior_z_qso_increase - 0.01
    no, lls, dla = MO.multi_priors(prior["z_qsos"], prior["dla_ind"], z_low, 4, Z_lls, Z_dla)
    assert np.isnan(no) and np.isnan(lls) and np.all(np.isnan(dla))


# ------------------------------------------------------------------------------------------------ the kernels (GPU)
def _multi(api, model, samples, spectra, prior, base=None, **kw):
    return api.process_qsos_multiple_dlas_meanflux(model, samples, spectra, prior, base_sample_inds=base, **kw)


def _model(synthetic_inputs, k):
    from gp_dla_detection_b200 import synthetic as syn
    return synthetic_inputs["model"] if k == 20 else syn.make_model(k)


@gpu
@pytest.mark.parametrize("k", [20, 40])
def test_split_batches_against_oracle(api, synthetic_inputs, monkeypatch, k):
    """A batch of >= 148 quasars puts its last ~7 % on the FP64 DMMA kernels on the side stream, in all three modes
    of the fused kernels.  Every output of every quasar must be the bits of the path that processed it, and the split
    run must match the oracle.  k = 20 runs the default batches (148 split, then 4 whole on INT8); k = 40 one batch
    of all quasars.  An empty spectrum and a quasar forced to stop after level 1 sit in each share."""
    from gp_dla_detection_b200 import synthetic as syn
    si = synthetic_inputs
    model = _model(si, k)
    Q, S = 152, 40
    samples = syn.make_samples(S, with_lls=True)
    sp = syn.make_spectra(model, Q, seed=210 + k, dla_fraction=0.6, meanflux=True, second_dla_fraction=0.5)
    batch = 148 if k == 20 else Q
    n2 = int(round(0.072 * batch))
    on_f64 = np.zeros(Q, dtype=bool)
    on_f64[batch - n2:batch] = True
    empty = [5, batch - 3] + ([Q - 1] if batch < Q else [])
    forced = [7, batch - 5] + ([Q - 3] if batch < Q else [])
    for q in empty:
        sp["all_pixel_mask"][q][:] = True
    own = _oracle(model, samples, sp, si["prior"])
    base, ref = _force_early_exit(model, samples, sp, si["prior"], own, forced)
    bq = 0 if k == 20 else Q
    split = _multi(api, model, samples, sp, si["prior"], base, batch_quasars=bq)
    monkeypatch.setenv("GPDLA_F64_SHARE", "0")
    whole = _multi(api, model, samples, sp, si["prior"], base, batch_quasars=bq)
    monkeypatch.delenv("GPDLA_F64_SHARE")
    f64 = _multi(api, model, samples, sp, si["prior"], base, batch_quasars=bq, gram_digits=-1)
    assert_multi_parity(split, ref)
    assert_same(split, whole, ~on_f64)
    assert_same(split, f64, on_f64)
    # the two paths round differently, so a quasar computed by the wrong one would show
    a, w = split["sample_log_likelihoods_dla"], whole["sample_log_likelihoods_dla"]
    assert not np.array_equal(a[on_f64], w[on_f64], equal_nan=True)
    assert np.allclose(a, w, rtol=1e-11, atol=0, equal_nan=True)
    for q in forced:
        _assert_stopped_after_level_1(split, q)
    for q in empty:
        assert np.all(np.isnan(split["log_likelihoods_dla"][q])) and np.all(split["MAP_inds"][q] == -1)
    others = np.setdiff1d(np.arange(Q), forced + empty)
    assert np.all(np.isfinite(split["log_likelihoods_dla"][others, 0]))
    assert np.any(np.isfinite(split["log_likelihoods_dla"][others[others < batch - n2], 3]))
    assert np.any(np.isfinite(split["log_likelihoods_dla"][np.intersect1d(others, np.flatnonzero(on_f64)), 1]))
    if k == 20:   # the built-in resampling once against the oracle's (a draw within ~1e-13 of an edge may differ)
        res = _multi(api, model, samples, sp, si["prior"])
        same = np.mean(res["base_sample_inds"] == own["base_sample_inds"])
        assert same > 0.999, same


@gpu
def test_single_dla_split_at_rank_40(api, synthetic_inputs, monkeypatch):
    """The same split on the single-DLA path at k = 40 (column-split kernels and the stand-alone Cholesky), which a
    batch of >= 148 quasars reaches."""
    from gp_dla_detection_b200 import synthetic as syn
    from oracle import process_qsos_oracle as O
    from test_gpu_parity import assert_parity
    si = synthetic_inputs
    m40 = syn.make_model(40)
    Q = 152
    samples = syn.make_samples(40)
    sp = syn.make_spectra(m40, Q, seed=220, dla_fraction=0.5)
    sp["all_pixel_mask"][3][:] = True
    sp["all_pixel_mask"][145][:] = True

    def run(**kw):
        proc = api.DLAProcessor(m40, samples, si["prior"], batch_quasars=Q, **kw)
        try:
            return proc.process(sp)
        finally:
            proc.close()

    split = run()
    monkeypatch.setenv("GPDLA_F64_SHARE", "0")
    whole = run()
    monkeypatch.delenv("GPDLA_F64_SHARE")
    f64 = run(gram_digits=-1)
    n2 = int(round(0.072 * Q))
    assert_same(split, whole, slice(0, Q - n2))
    assert_same(split, f64, slice(Q - n2, Q))
    assert not np.array_equal(split["sample_log_likelihoods_dla"][Q - n2:], whole["sample_log_likelihoods_dla"][Q - n2:],
                              equal_nan=True)
    assert_parity(split, O.process_qsos(m40, samples, sp, si["prior"], engine="c"))


@gpu
@pytest.mark.parametrize("k", [20, 40])
def test_fp64_fallback_list_in_every_mode(api, synthetic_inputs, k):
    """Used pixels with zero noise variance send a quasar from the INT8 kernels to the FP64 list kernels, which then
    write (mode 1) and read (mode 2) the absorption cache for it.  Against the oracle; the other quasars keep the
    bits of a run without the flagged ones; more flagged quasars than the list launch has slots."""
    from gp_dla_detection_b200 import synthetic as syn
    si = synthetic_inputs
    model = _model(si, k)
    samples = syn.make_samples(64, with_lls=True)
    sp = syn.make_spectra(model, 4, seed=230 + k, dla_fraction=0.75, meanflux=True, second_dla_fraction=0.5)
    for q in (1, 3):
        _zero_noise(sp, q, [-3, -11, -12, -24])
    ref = _oracle(model, samples, sp, si["prior"])
    res = _multi(api, model, samples, sp, si["prior"], ref["base_sample_inds"])
    assert np.all(np.isfinite(res["sample_log_likelihoods_dla"][:, :, 0]))
    assert_multi_parity(res, ref)
    clean = _multi(api, model, samples, _quasars(sp, [0, 2]), si["prior"], ref["base_sample_inds"][[0, 2]])
    assert_same(_rows(res, [0, 2]), clean)
    samples3 = syn.make_samples(40, with_lls=True)
    sp3 = syn.make_spectra(model, 11, seed=240 + k, dla_fraction=0.5, meanflux=True, second_dla_fraction=0.5)
    for q in range(11):
        _zero_noise(sp3, q, [-2 - q])
    ref3 = _oracle(model, samples3, sp3, si["prior"])
    assert_multi_parity(_multi(api, model, samples3, sp3, si["prior"], ref3["base_sample_inds"]), ref3)


@gpu
def test_rank_arithmetic_lines_and_levels(api, synthetic_inputs):
    """k = 10 (FP64 only); k = 20 on every Gram arithmetic with and without the rest-frame table; 1, 5 and 31 lines
    (the run-time line-count kernels) and 1, 2 or 4 levels on both Gram paths."""
    from gp_dla_detection_b200 import synthetic as syn
    from gp_dla_detection_b200.params import Parameters
    si = synthetic_inputs
    samples = syn.make_samples(48, with_lls=True)
    m10 = syn.make_model(10)
    sp10 = syn.make_spectra(m10, 3, seed=250, dla_fraction=0.7, meanflux=True, second_dla_fraction=0.5)
    ref = _oracle(m10, samples, sp10, si["prior"])
    assert_multi_parity(_multi(api, m10, samples, sp10, si["prior"], ref["base_sample_inds"]), ref)
    model = si["model"]
    sp = syn.make_spectra(model, 3, seed=251, dla_fraction=0.7, meanflux=True, second_dla_fraction=0.5)
    ref = _oracle(model, samples, sp, si["prior"])
    for digits in (6, 5, -1):
        for rest_table in (0, -1):
            res = _multi(api, model, samples, sp, si["prior"], ref["base_sample_inds"], gram_digits=digits,
                         rest_table=rest_table)
            assert_multi_parity(res, ref, ll_rtol=1e-9 if digits == 5 else LL_RTOL)
    for nl in (1, 5, 31):
        ref = _oracle(model, samples, sp, si["prior"], num_lines=nl)
        for digits in (0, -1):
            res = _multi(api, model, samples, sp, si["prior"], ref["base_sample_inds"], gram_digits=digits,
                         params=Parameters(num_lines=nl))
            assert_multi_parity(res, ref)
    for md in (1, 2, 4):
        ref = _oracle(model, samples, sp, si["prior"], max_dlas=md)
        for digits in (0, -1):
            res = _multi(api, model, samples, sp, si["prior"], ref["base_sample_inds"] if md > 1 else None,
                         max_dlas=md, gram_digits=digits)
            assert res["model_posteriors"].shape == (3, md + 2)
            assert_multi_parity(res, ref)


@gpu
@pytest.mark.parametrize("k,S", [(20, 1), (20, 5), (20, 33), (20, 127), (20, 129), (20, 300),
                                 (40, 1), (40, 127), (40, 129)])
def test_sample_counts(api, synthetic_inputs, k, S):
    """Partial tiles, the null-model slot next to partner rows, resampling over a few samples.  At S = 1 the only
    partner of the only sample is itself: levels 2-4 are NaN and so are the posteriors."""
    from gp_dla_detection_b200 import synthetic as syn
    si = synthetic_inputs
    model = _model(si, k)
    samples = syn.make_samples(S, with_lls=True)
    sp = syn.make_spectra(model, 2, seed=260 + k, dla_fraction=1.0, meanflux=True, second_dla_fraction=0.5)
    ref = _oracle(model, samples, sp, si["prior"])
    for digits in (0, -1):
        res = _multi(api, model, samples, sp, si["prior"], ref["base_sample_inds"], gram_digits=digits)
        assert_multi_parity(res, ref)
    if S == 1:
        res = _multi(api, model, samples, sp, si["prior"])                   # the built-in resampling too
        assert_multi_parity(res, ref)
        for q in range(2):
            _assert_stopped_after_level_1(res, q)
            assert np.all(np.isnan(res["model_posteriors"][q]))


@gpu
@pytest.mark.parametrize("digits", [0, -1])
def test_sample_permutation_with_mapped_partners(api, synthetic_inputs, digits):
    """The kernels walk samples sorted by offset: the absorption cache is indexed by sample, the tiles by position.
    Permuting the samples and mapping the partners through the permutation must permute the sample log-likelihoods
    bit for bit and map the MAP through the permutation."""
    from gp_dla_detection_b200 import synthetic as syn
    si = synthetic_inputs
    S = 300
    samples = syn.make_samples(S, with_lls=True)
    sp = syn.make_spectra(si["model"], 3, seed=270, dla_fraction=1.0, meanflux=True, second_dla_fraction=1.0)
    base = _multi(api, si["model"], samples, sp, si["prior"], gram_digits=digits)["base_sample_inds"]
    a = _multi(api, si["model"], samples, sp, si["prior"], base, gram_digits=digits)
    perm = np.random.default_rng(4).permutation(S)
    sperm = {k: (v[perm] if np.ndim(v) else v) for k, v in samples.items()}
    b = _multi(api, si["model"], sperm, sp, si["prior"], np.argsort(perm)[base[:, perm, :]], gram_digits=digits)
    sa, sb = a["sample_log_likelihoods_dla"], b["sample_log_likelihoods_dla"]
    assert np.array_equal(sa[:, perm, :], sb, equal_nan=True)
    assert np.array_equal(a["sample_log_likelihoods_lls"][:, perm], b["sample_log_likelihoods_lls"])
    for k in ("log_likelihoods_dla", "log_likelihoods_lls", "log_posteriors_dla"):
        assert np.allclose(a[k], b[k], rtol=LEVEL_RTOL, atol=0, equal_nan=True), k
    assert np.allclose(a["model_posteriors"], b["model_posteriors"], rtol=0, atol=1e-12, equal_nan=True)
    assert np.isfinite(a["log_likelihoods_dla"][:, 1]).all()
    for q in range(3):
        for l in range(4):
            i, j = a["MAP_inds"][q, l, 0], b["MAP_inds"][q, l, 0]
            assert (i < 0) == (j < 0), (q, l)
            if i < 0:
                continue
            if perm[j] == i:
                assert np.array_equal(perm[b["MAP_inds"][q, l, :l + 1]], a["MAP_inds"][q, l, :l + 1])
                assert np.array_equal(a["MAP_z_dlas"][q, l], b["MAP_z_dlas"][q, l], equal_nan=True)
            else:   # an exact tie: the same absorbers in another order
                assert l >= 1 and sa[q, i, l] == sb[q, j, l], (q, l)


@gpu
@pytest.mark.parametrize("digits", [0, -1])
def test_early_exit_in_a_running_batch(api, synthetic_inputs, digits):
    """Quasars that stop after level 1 next to quasars that go on to level 4, on each Gram path and at k = 40."""
    from gp_dla_detection_b200 import synthetic as syn
    si = synthetic_inputs
    samples = syn.make_samples(48, with_lls=True)
    for k in (20, 40):
        model = _model(si, k)
        sp = syn.make_spectra(model, 5, seed=280 + k, dla_fraction=0.6, meanflux=True, second_dla_fraction=0.5)
        own = _oracle(model, samples, sp, si["prior"])
        base, ref = _force_early_exit(model, samples, sp, si["prior"], own, [1, 3])
        res = _multi(api, model, samples, sp, si["prior"], base, gram_digits=digits)
        assert_multi_parity(res, ref)
        for q in (1, 3):
            _assert_stopped_after_level_1(res, q)
        assert np.any(np.isfinite(res["log_likelihoods_dla"][[0, 2, 4], 3]))


@gpu
def test_prior_edges(api, synthetic_inputs):
    """Catalogues without DLAs, with nothing but DLAs, and a quasar below every catalogue redshift: the +-inf / NaN
    patterns of every prior, posterior and p_* output, on both paths (prepare_quasars_kernel counts the prior for
    both)."""
    from gp_dla_detection_b200 import synthetic as syn
    from oracle import process_qsos_multi_oracle as MO
    from oracle import process_qsos_oracle as O
    from test_gpu_parity import assert_parity
    si = synthetic_inputs
    samples = syn.make_samples(40, with_lls=True)
    sp = syn.make_spectra(si["model"], 3, seed=290, dla_fraction=0.7, meanflux=True)
    z_low = float(np.min(si["prior"]["z_qsos"])) - O.prior_z_qso_increase - 0.02
    sp["all_wavelengths"][2] = sp["all_wavelengths"][2] * (1 + z_low) / (1 + float(sp["z_qsos"][2]))
    sp["z_qsos"][2] = z_low                                                  # the same rest frame, below the catalogue
    base = None
    for name, prior in _edge_priors(si["prior"]).items():
        ref = _oracle(si["model"], samples, sp, prior, base_sample_inds=base)
        base = ref["base_sample_inds"]
        res = _multi(api, si["model"], samples, sp, prior, base)
        assert_multi_parity(res, ref)
        for q in range(3):
            no, lls, dla = MO.multi_priors(prior["z_qsos"], prior["dla_ind"], float(sp["z_qsos"][q]), 4,
                                           samples["Z_lls"], samples["Z_dla"])
            got = np.concatenate([[res["log_priors_no_dla"][q], res["log_priors_lls"][q]], res["log_priors_dla"][q]])
            assert np.allclose(got, np.concatenate([[no, lls], dla]), rtol=1e-13, atol=0, equal_nan=True), (name, q)
        for key in ("log_priors_no_dla", "log_priors_lls", "log_priors_dla", "log_posteriors_no_dla",
                    "log_posteriors_lls", "log_posteriors_dla", "model_posteriors", "p_no_dlas", "p_lls", "p_dlas"):
            for f in (np.isnan, np.isposinf, np.isneginf):
                assert np.array_equal(f(res[key]), f(ref[key])), (name, key)
        assert np.all(np.isnan(res["model_posteriors"][2])) and np.isnan(res["log_priors_no_dla"][2])
        if name == "no_dlas":   # -inf priors: the null model takes everything (unless a level stopped: NaN)
            for q in np.flatnonzero(np.all(np.isfinite(ref["log_likelihoods_dla"][:2]), axis=1)):
                assert np.array_equal(res["model_posteriors"][q], [1.0, 0, 0, 0, 0, 0])
        single = api.process_qsos(si["model"], samples, sp, prior)
        assert_parity(single, O.process_qsos(si["model"], samples, sp, prior, engine="c"))


def _extreme_spectra(model, rng):
    from gp_dla_detection_b200 import synthetic as syn
    sp = syn.make_spectra(model, 12, seed=300, dla_fraction=0.6, meanflux=True, second_dla_fraction=0.5)
    for q in range(12):
        L = len(sp["all_flux"][q])
        sp["all_noise_variance"][q] = 10.0 ** rng.uniform(-6, 4, L)
        sp["all_flux"][q] = sp["all_flux"][q] + rng.standard_normal(L) * np.sqrt(sp["all_noise_variance"][q])
        out = rng.random(L) < 0.01
        sp["all_flux"][q][out] = rng.uniform(-50, 50, np.count_nonzero(out))
        sp["all_pixel_mask"][q] = rng.random(L) < rng.choice([0.0, 0.05, 0.5])
        if q % 4 == 0:
            lo, n_keep = rng.integers(0, 900), rng.integers(210, 400)
            for k in ("all_wavelengths", "all_flux", "all_noise_variance", "all_pixel_mask"):
                sp[k][q] = sp[k][q][lo:lo + n_keep]
    sp["all_wavelengths"][3] = sp["all_wavelengths"][3] * (1 + 5.5) / (1 + float(sp["z_qsos"][3]))   # all 31 lines
    sp["z_qsos"][3] = 5.5
    return sp


@gpu
def test_ragged_masked_and_extreme_spectra(api, synthetic_inputs):
    """Trimmed blue and red ends, NaN flux under the mask, an empty spectrum; then noise variances over 10 decades,
    flux outliers, heavy masking, short spectra and a quasar at z = 5.5, MAP checked where it is tie-free."""
    from gp_dla_detection_b200 import synthetic as syn
    si = synthetic_inputs
    model = si["model"]
    samples = syn.make_samples(40, with_lls=True)
    sp = syn.make_spectra(model, 4, seed=310, dla_fraction=0.7, meanflux=True, second_dla_fraction=0.5)
    for k in ("all_wavelengths", "all_flux", "all_noise_variance", "all_pixel_mask"):
        sp[k][0] = sp[k][0][500:]                      # blue end missing
        sp[k][2] = sp[k][2][:900]                      # red end missing
    sp["all_pixel_mask"][1][200:260] = True
    sp["all_flux"][1][200:260] = np.nan                # garbage under the mask must not leak
    sp["all_pixel_mask"][3][:] = True
    spo = _quasars(sp, [0, 1, 2, 3])
    spo["all_flux"][1] = np.where(sp["all_pixel_mask"][1], 0.0, sp["all_flux"][1])
    ref = _oracle(model, samples, spo, si["prior"])
    for digits in (0, -1):
        res = _multi(api, model, samples, sp, si["prior"], ref["base_sample_inds"], gram_digits=digits)
        assert_multi_parity(res, ref)
        assert np.all(np.isnan(res["log_likelihoods_dla"][3])) and np.isnan(res["log_likelihoods_lls"][3])

    sp = _extreme_spectra(model, np.random.default_rng(2024))
    ref = _oracle(model, samples, sp, si["prior"])
    b = ref["sample_log_likelihoods_dla"]
    for digits in (0, -1):
        res = _multi(api, model, samples, sp, si["prior"], ref["base_sample_inds"], gram_digits=digits)
        assert_multi_parity(res, ref, ll_rtol=1e-9, check_map=False)
        for q in range(12):
            for l in range(4):
                col = b[q, :, l]
                if np.all(np.isnan(col)):
                    assert res["MAP_inds"][q, l, 0] == -1
                    continue
                m = np.nanmax(col)
                if np.sum(col >= m - 2e-9 * abs(m)) == 1:                    # tie-free at the values' own bar
                    assert np.array_equal(res["MAP_inds"][q, l], ref["MAP_inds"][q, l]), (q, l)


@gpu
def test_entries_outputs_and_workspace_reuse(api, synthetic_inputs):
    """Several batches, no large outputs (host and device entries), the device entry with given indices, and one
    context alternating single- and multi-DLA calls of other L_max, level and batch counts: each gives the bits of the
    plain host run with the same indices."""
    import torch
    from gp_dla_detection_b200 import synthetic as syn
    si = synthetic_inputs
    model, prior = si["model"], si["prior"]
    samples = syn.make_samples(64, with_lls=True)
    sp = syn.make_spectra(model, 7, seed=320, dla_fraction=0.6, meanflux=True, second_dla_fraction=0.5)
    sp["all_pixel_mask"][4][:] = True
    plain = _multi(api, model, samples, sp, prior)
    base = plain["base_sample_inds"]
    ref = _multi(api, model, samples, sp, prior, base)
    assert_same(ref, plain)
    assert_same(_multi(api, model, samples, sp, prior, base, batch_quasars=2), ref)
    small = _multi(api, model, samples, sp, prior, base, return_samples=False)
    assert set(ref) - set(small) == {"sample_log_likelihoods_dla", "sample_log_likelihoods_lls", "base_sample_inds"}
    assert_same(small, {k: ref[k] for k in small})
    assert_same(_multi(api, model, samples, sp, prior, return_samples=False), small)   # same draws without the arrays

    pad = api.pad_spectra(sp)
    t = {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in pad.items()}
    planes = (t["wavelengths"], t["flux"], t["noise_variance"], t["pixel_mask"], t["lengths"], t["z_qsos"])
    proc = api.DLAProcessor(model, samples, prior, batch_quasars=3)
    try:
        bt = torch.from_numpy(np.ascontiguousarray(np.transpose(base, (0, 2, 1)), dtype=np.int32)).cuda()
        for want in (True, False):
            dev = proc.process_multi_device(*planes, max_dlas=4, base_sample_inds=bt, return_samples=want)
            torch.cuda.synchronize()
            got = {k: v.cpu().numpy() for k, v in dev.items()}
            if want:
                for k in ("sample_log_likelihoods_dla", "base_sample_inds"):
                    got[k] = np.transpose(got[k], (0, 2, 1))
            assert_same(got, {k: ref[k] for k in got})
    finally:
        proc.close()

    # one context, alternating entries, L_max, levels and batch sizes, against fresh contexts
    fixed = syn.make_spectra(model, 3, seed=321, fixed_shape=True, dla_fraction=0.6, meanflux=True)
    single = syn.make_spectra(model, 5, seed=322, dla_fraction=0.5)
    fresh_single = api.process_qsos(model, samples, single, prior)
    fresh_fixed_single = api.process_qsos(model, samples, fixed, prior)
    fresh_fixed = _multi(api, model, samples, fixed, prior, max_dlas=2)
    base2 = fresh_fixed["base_sample_inds"]
    proc = api.DLAProcessor(model, samples, prior)
    try:
        for _ in range(2):                                                   # the second round repeats every call
            assert_same(proc.process(single), fresh_single)
            assert_same(proc.process_multi(sp, 4, base), ref)
            assert_same(proc.process(fixed), fresh_fixed_single)
            assert_same(proc.process_multi(fixed, 2, base2), fresh_fixed)
            assert_same(proc.process_multi(_quasars(sp, [6, 0]), 3, base[[6, 0]][:, :, :2]),
                        _multi(api, model, samples, _quasars(sp, [6, 0]), prior, base[[6, 0]][:, :, :2], max_dlas=3))
    finally:
        proc.close()
