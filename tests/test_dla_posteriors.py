"""Per-quasar absorber posterior summaries (effective sample size, moments, credible intervals, DLA-threshold mass): the
NumPy restatement pinned by hand values on the CPU, the C entries' argument checks, the sharded gather, and on the GPU
the kernels against the restatement, a simulation-based calibration and an end-to-end run."""
import ctypes
import math
import os
import socket

import numpy as np
import pytest

from gp_dla_detection_b200 import _lib, api
from gp_dla_detection_b200 import sharding as sh
from oracle import dla_posteriors_oracle as O

OFF = np.array([0.1, 0.6, 0.3, 0.9, 0.05])                 # z = 2.1, 2.6, 2.3, 2.9, 2.05 for z in [2, 3]
LNHI = np.array([20.0, 20.5, 21.5, 20.35, 19.5])


# ------------------------------------------------------------------ the restatement, by hand
def test_oracle_one_sample_with_all_the_weight():
    ll = np.array([-np.inf, 0.0, -1e4, np.nan, -800.0])        # exp(-800) underflows: sample 1 carries everything
    rec = O.quasar_posterior(ll, 2.0, 3.0, OFF, LNHI, [0.01, 0.5, 0.99], threshold=20.3)
    z1 = 2.0 + (3.0 - 2.0) * 0.6
    assert rec[0] == 1.0
    assert rec[1] == z1 and rec[2] == 0.0 and rec[3] == 20.5 and rec[4] == 0.0 and rec[5] == 0.0
    assert rec[6] == 1.0
    assert np.all(rec[7:10] == z1) and np.all(rec[10:13] == 20.5)


def test_oracle_two_equal_weights_lower_quantile():
    ll = np.array([-np.inf, 0.0, 0.0, -np.inf, np.nan])        # samples 1 (z 2.6, 20.5) and 2 (z 2.3, 21.5)
    eps = 1e-9
    rec = O.quasar_posterior(ll, 2.0, 3.0, OFF, LNHI, [0.5, 0.5 + eps], threshold=21.0)
    za, zb = 2.0 + 0.3, 2.0 + 0.6
    assert rec[0] == 2.0
    assert rec[7] == za and rec[8] == zb                       # p = 0.5 reaches the lower one, 0.5 + eps the upper
    assert rec[9] == 20.5 and rec[10] == 21.5
    assert rec[6] == 0.5
    assert abs(rec[1] - (za + zb) / 2) < 1e-15 and abs(rec[2] - (zb - za) / 2) < 1e-15
    assert abs(rec[5] - (-(zb - za) / 2 * 0.5)) < 1e-15         # z and log N move in opposite directions


@pytest.mark.parametrize("why", ["all_nan", "all_minus_inf", "plus_inf", "empty_z", "nan_z"])
def test_oracle_nan_record(why):
    ll, zlo, zhi = np.zeros(5), 2.0, 3.0
    if why == "all_nan":
        ll[:] = np.nan
    elif why == "all_minus_inf":
        ll[:] = -np.inf
    elif why == "plus_inf":
        ll[2] = np.inf
    elif why == "empty_z":
        zhi = 2.0
    else:
        zlo = np.nan
    rec = O.quasar_posterior(ll, zlo, zhi, OFF, LNHI, [0.5])
    assert rec.shape == (9,) and np.all(np.isnan(rec))


def test_oracle_moments_equal_np_average():
    rng = np.random.default_rng(2)
    S = 257
    off, lnhi = rng.random(S), rng.uniform(20.0, 22.5, S)
    ll = -0.5 * rng.standard_normal(S) ** 2 * 8
    ll[::17] = np.nan
    ll[5::31] = -np.inf
    rec = O.quasar_posterior(ll, 2.4, 3.3, off, lnhi, [0.3], threshold=21.0)
    ok = ll > -np.inf
    w = np.exp(ll[ok] - ll[ok].max())
    z = (2.4 + (3.3 - 2.4) * off)[ok]
    n = lnhi[ok]
    zm, nm = np.average(z, weights=w), np.average(n, weights=w)
    np.testing.assert_allclose(rec[[1, 3]], [zm, nm], rtol=1e-14)
    np.testing.assert_allclose(rec[[2, 4]], np.sqrt([np.average((z - zm) ** 2, weights=w),
                                                     np.average((n - nm) ** 2, weights=w)]), rtol=1e-12)
    np.testing.assert_allclose(rec[5], np.average((z - zm) * (n - nm), weights=w), rtol=1e-12)
    np.testing.assert_allclose(rec[0], w.sum() ** 2 / np.sum(w * w), rtol=1e-14)
    np.testing.assert_allclose(rec[6], np.average(n >= 21.0, weights=w), rtol=1e-14)


def test_multi_oracle_one_level_is_the_single_oracle():
    rng = np.random.default_rng(4)
    S = 300
    off, lnhi = rng.random(S), rng.uniform(20.0, 22.5, S)
    ll = -0.5 * rng.standard_normal((6, 1, S)) ** 2 * 5
    ll[1, 0, ::3] = np.nan
    zlo, zhi = rng.uniform(2.0, 3.0, 6), rng.uniform(2.0, 4.0, 6)   # some empty ranges
    multi = O.multi_dla_posteriors(ll, None, zlo, zhi, off, lnhi)
    single = O.dla_posteriors(ll[:, 0], zlo, zhi, off, lnhi, [0.5])
    assert multi.shape == (6, 5)
    assert np.array_equal(multi, single[:, :5], equal_nan=True)
    assert np.any(np.isnan(multi[:, 0])) and np.any(np.isfinite(multi[:, 0]))


def test_multi_oracle_ranks_are_ordered_and_levels_independent():
    rng = np.random.default_rng(5)
    S, J = 200, 4
    off, lnhi = rng.random(S), rng.uniform(20.0, 22.5, S)
    ll = -0.5 * rng.standard_normal((J, S)) ** 2 * 3
    part = rng.integers(0, S, (J - 1, S))
    rec = O.multi_quasar_posterior(ll, part, 2.2, 3.4, off, lnhi)
    t = api.unpack_multi_dla_posteriors(rec[None], J)
    for j in range(2, J + 1):
        zm = t["z_mean"][0, j - 1, :j]
        assert np.all(np.diff(zm) >= 0), zm                   # the rank-r z is pointwise ordered, so are the means
    # a poisoned partner in row 1 (used from level 3 on) makes levels 3 and 4 NaN only
    bad = part.copy()
    bad[1, 7] = S
    rec2 = O.multi_quasar_posterior(ll, bad, 2.2, 3.4, off, lnhi)
    t2 = api.unpack_multi_dla_posteriors(rec2[None], J)
    assert np.array_equal(t2["ess"][0, :2], t["ess"][0, :2]) and np.all(np.isnan(t2["ess"][0, 2:]))


def test_unpack_and_monte_carlo_spread():
    P = 2
    rec = np.array([[4.0, 2.5, 0.1, 21.0, 0.2, -0.01, 0.6, 2.4, 2.6, 20.8, 21.2],
                    [np.nan] * 11])
    t = api.unpack_dla_posteriors(rec, P, num_samples=100, p_dlas=[0.8, np.nan])
    assert t["z_quantiles"].tolist()[0] == [2.4, 2.6] and t["log_nhi_quantiles"].tolist()[0] == [20.8, 21.2]
    assert t["mass_above_threshold"][0] == 0.6
    assert t["log_likelihood_dla_mc_sd"][0] == math.sqrt(1 / 4 - 1 / 100)
    assert t["p_dla_mc_sd"][0] == 0.8 * (1 - 0.8) * math.sqrt(1 / 4 - 1 / 100)
    assert np.isnan(t["p_dla_mc_sd"][1])
    assert api.unpack_dla_posteriors(np.array([[100.0] + [0.0] * 8]), 1, num_samples=100)["log_likelihood_dla_mc_sd"][0] == 0
    with pytest.raises(ValueError):
        api.unpack_dla_posteriors(rec, 3)


# ------------------------------------------------------------------ the C entries' argument checks (no GPU needed)
def _call_single(device=False, Q=1, S=4, quantiles=(0.5,), P=None, threshold=20.3, null=None):
    lib = _lib.load()
    n, s = min(max(Q, 1), 4), max(S, 1)                        # the arrays of an accepted call; the rest is checked
    ll, zlo, zhi = np.zeros((n, s)), np.full(n, 2.0), np.full(n, 3.0)
    off, lnhi = np.linspace(0, 1, s), np.full(s, 21.0)
    qs = np.asarray(quantiles, dtype=np.float64)
    out = np.zeros((n, 7 + 2 * max(qs.size, 1)))
    vp = lambda a, n: None if null == n else ctypes.c_void_p(a.ctypes.data)
    args = [Q, S, vp(ll, "ll"), vp(zlo, "zlo"), vp(zhi, "zhi"), vp(off, "off"), vp(lnhi, "lnhi"),
            qs.size if P is None else P, None if null == "quantiles" else api._dp(qs), threshold, vp(out, "out")]
    rc = lib.gpdla_dla_posteriors_device(*args, None) if device else lib.gpdla_dla_posteriors(*args)
    return rc, (lib.gpdla_last_error(None) or b"").decode()


def _call_multi(device=False, Q=1, S=4, max_dlas=3, null=None):
    lib = _lib.load()
    J, n, s = min(max(max_dlas, 1), 4), min(max(Q, 1), 4), max(S, 1)
    ll, part = np.zeros((n, J, s)), np.zeros((n, max(J - 1, 1), s), dtype=np.int32)
    zlo, zhi, off, lnhi = np.full(n, 2.0), np.full(n, 3.0), np.linspace(0, 1, s), np.full(s, 21.0)
    out = np.zeros((n, J + 2 * J * (J + 1)))
    vp = lambda a, n: None if null == n else ctypes.c_void_p(a.ctypes.data)
    args = [Q, S, max_dlas, vp(ll, "ll"), vp(part, "part"), vp(zlo, "zlo"), vp(zhi, "zhi"), vp(off, "off"),
            vp(lnhi, "lnhi"), vp(out, "out")]
    rc = lib.gpdla_multi_dla_posteriors_device(*args, None) if device else lib.gpdla_multi_dla_posteriors(*args)
    return rc, (lib.gpdla_last_error(None) or b"").decode()


SINGLE_BAD = dict(no_quantiles=dict(quantiles=(), P=0), seventeen=dict(quantiles=np.full(17, 0.5)),
                  p_zero=dict(quantiles=(0.0, 0.5)), p_one=dict(quantiles=(0.5, 1.0)), p_nan=dict(quantiles=(np.nan,)),
                  p_negative=dict(quantiles=(-0.1,)), threshold_nan=dict(threshold=np.nan),
                  threshold_inf=dict(threshold=np.inf), negative_q=dict(Q=-1), zero_s=dict(S=0),
                  big_q=dict(Q=2 ** 31), null_ll=dict(null="ll"), null_out=dict(null="out"),
                  null_offsets=dict(null="off"), null_quantiles=dict(null="quantiles"))


@pytest.mark.parametrize("device", [False, True])
@pytest.mark.parametrize("case", sorted(SINGLE_BAD))
def test_c_entry_rejects_bad_arguments(case, device):
    rc, msg = _call_single(device=device, **SINGLE_BAD[case])
    assert rc == _lib.GPDLA_ERR_INVALID, (rc, msg)
    name = "gpdla_dla_posteriors_device" if device else "gpdla_dla_posteriors"
    assert msg.startswith(name + ": "), msg


MULTI_BAD = dict(max_dlas_zero=dict(max_dlas=0), max_dlas_five=dict(max_dlas=5), null_partners=dict(null="part"),
                 null_ll=dict(null="ll"), null_log_nhi=dict(null="lnhi"), zero_s=dict(S=0), negative_q=dict(Q=-1))


@pytest.mark.parametrize("device", [False, True])
@pytest.mark.parametrize("case", sorted(MULTI_BAD))
def test_multi_c_entry_rejects_bad_arguments(case, device):
    rc, msg = _call_multi(device=device, **MULTI_BAD[case])
    assert rc == _lib.GPDLA_ERR_INVALID, (rc, msg)
    name = "gpdla_multi_dla_posteriors_device" if device else "gpdla_multi_dla_posteriors"
    assert msg.startswith(name + ": "), msg


def test_entries_accept_the_limits():
    """16 quantiles, one level without partners, and Q = 0 pass the checks (a non-empty call then needs a device)."""
    import torch
    want = _lib.GPDLA_OK if torch.cuda.is_available() else _lib.GPDLA_ERR_CUDA
    rc, msg = _call_single(quantiles=np.linspace(0.01, 0.99, 16))
    assert rc == want, msg
    rc, msg = _call_multi(max_dlas=1, null="part")
    assert rc == want, msg
    rc, msg = _call_single(device=True, Q=0, null="ll")
    assert rc == _lib.GPDLA_OK, msg


# ------------------------------------------------------------------ sharded gather, 2 gloo ranks, CPU stand-in
S_STAND_IN, QUANTILES = 64, (0.1, 0.5, 0.9)


def _stand_in_samples(S=S_STAND_IN):
    return (np.arange(S) + 0.5) / S, 20.0 + 3.0 * ((np.arange(S) * 0.618034) % 1.0)


def _stand_in_records(sp):
    """Oracle records of deterministic stand-ins for process_device outputs, keyed on z_qso."""
    z = np.asarray(sp["z_qsos"])
    off, lnhi = _stand_in_samples()
    ll = -50.0 * (off[None, :] - np.modf(7.0 * z)[0][:, None]) ** 2
    return O.dla_posteriors(ll, z - 1.0, z - 0.05, off, lnhi, QUANTILES)


def _posteriors_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from gp_dla_detection_b200 import synthetic as syn
    spectra = syn.make_spectra(syn.make_model(), 11, seed=6)
    res = sh.dla_posteriors_sharded(None, None, spectra, None, quantiles=QUANTILES, batch_quasars=2,
                                    compute=_stand_in_records)
    q.put((rank, res["records"].tobytes(), res["records"].shape, res["blocks"]))
    dist.destroy_process_group()


def test_sharded_posteriors_two_gloo_ranks():
    import torch.multiprocessing as mp
    from gp_dla_detection_b200 import synthetic as syn
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_posteriors_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    results = sorted(q.get(timeout=180) for _ in range(2))
    for p in procs:
        p.join(60)
    (r0, b0, shape, blocks), (r1, b1, _, _) = results
    assert (r0, r1) == (0, 1) and b0 == b1
    assert blocks[0][1] > 0 and blocks[1][1] > blocks[0][1]       # both ranks hold quasars
    got = np.frombuffer(b0, dtype=np.float64).reshape(shape)
    ref = _stand_in_records(syn.make_spectra(syn.make_model(), 11, seed=6))
    assert got.shape == (11, api.dla_posteriors_width(len(QUANTILES)))
    assert np.array_equal(got, ref, equal_nan=True)               # catalogue order, the bits of every quasar
    assert np.all(np.isfinite(got))


# ------------------------------------------------------------------ on the GPU
def _up(a, dt):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, dtype=dt)).cuda()


def _planes(spectra):
    pad = api.pad_spectra(spectra)
    return (_up(pad["wavelengths"], np.float64), _up(pad["flux"], np.float64), _up(pad["noise_variance"], np.float64),
            _up(pad["pixel_mask"], np.uint8), _up(pad["lengths"], np.int32), _up(pad["z_qsos"], np.float64))


@pytest.fixture(scope="module")
def processed():
    """process_device outputs of 300 synthetic quasars with the 10 000 default samples."""
    from gp_dla_detection_b200 import synthetic as syn
    model = syn.make_model()
    samples = syn.make_samples(10000)
    proc = api.DLAProcessor(model, samples, syn.make_prior(), device=0)
    out = proc.process_device(*_planes(syn.make_spectra(model, 300, seed=11, dla_fraction=0.3)),
                              return_sample_log_likelihoods=True)
    host = {k: v.cpu().numpy() for k, v in out.items()}
    yield dict(proc=proc, samples=samples, out=out, host=host)
    proc.close()


def _scaled_close(g, r, rtol, floor=0.0):
    return np.abs(g - r) <= rtol * np.abs(r) + floor


def assert_matches_oracle(got, ll, zlo, zhi, off, lnhi, quantiles, threshold=20.3, rtol=1e-12):
    """Moments, ess and mass to rtol; every quantile one of the values the oracle's cumulative sums allow (the
    first-reaching sample, or a neighbour where |cumsum - p total| <= 1e-12 total).  Returns the ambiguous count."""
    P = len(quantiles)
    ref = O.dla_posteriors(ll, zlo, zhi, off, lnhi, quantiles, threshold)
    assert got.shape == ref.shape
    assert np.array_equal(np.isnan(got), np.isnan(ref))
    f = np.isfinite(ref[:, 0])
    g, r = got[f], ref[f]
    for c in (0, 1, 3, 6):                                      # ess, means, mass
        bad = ~_scaled_close(g[:, c], r[:, c], rtol, 1e-15 if c == 6 else 0.0)
        assert not np.any(bad), (O.FIELDS[c], g[bad, c][:3], r[bad, c][:3])
    # a deviation is known to the rounding of the values: standard deviations and the covariance get an ulp-scale floor
    for c, m in ((2, 1), (4, 3)):
        bad = ~_scaled_close(g[:, c], r[:, c], rtol, 4e-16 * np.abs(r[:, m]))
        assert not np.any(bad), (O.FIELDS[c], g[bad, c][:3], r[bad, c][:3])
    floor = 4e-16 * (np.abs(r[:, 1]) * r[:, 4] + np.abs(r[:, 3]) * r[:, 2])
    assert np.all(_scaled_close(g[:, 5], r[:, 5], rtol, floor)), "z_log_nhi_cov"
    ambiguous = 0
    z_all = lambda q: O.sample_z(zlo[q], zhi[q], off)
    for i, q in enumerate(np.flatnonzero(f)):
        w = O.weights(ll[q])
        for k, p in enumerate(quantiles):
            for vals, col in ((z_all(q), 7 + k), (np.asarray(lnhi, float), 7 + P + k)):
                ok, amb = O.acceptable_quantiles(vals, w, p)
                ambiguous += amb
                assert got[q, col] in ok, (q, p, col, got[q, col], ok, ref[q, col])
                if not amb:
                    assert got[q, col] == ref[q, col]
    return ambiguous


@pytest.mark.gpu
@pytest.mark.parametrize("P", [1, 5, 16])
def test_kernel_matches_oracle_on_processed_quasars(processed, P):
    rng = np.random.default_rng(P)
    host, samples, proc = processed["host"], processed["samples"], processed["proc"]
    qs = (0.5,) if P == 1 else api.DEFAULT_QUANTILES if P == 5 else tuple(rng.uniform(0.005, 0.995, P))
    thr = 20.3 if P != 16 else float(samples["log_nhi_samples"][123])   # a threshold on a stored sample value
    got = proc.posteriors_device(processed["out"], quantiles=qs, log_nhi_threshold=thr).cpu().numpy()
    amb = assert_matches_oracle(got, host["sample_log_likelihoods_dla"], host["min_z_dlas"], host["max_z_dlas"],
                                samples["offset_samples"], samples["log_nhi_samples"], qs, thr)
    nfinite = int(np.count_nonzero(np.isfinite(got[:, 0])))
    print("P = %d: %d of %d quasars summarised; %d quantiles where a neighbour was within 1e-12 of the target"
          % (P, nfinite, got.shape[0], amb))
    assert nfinite > 0.9 * got.shape[0]


@pytest.mark.gpu
def test_large_sample_count_through_l2():
    """S = 100 000 does not fit in shared memory: every pass reads the row through the permutation."""
    from gp_dla_detection_b200 import synthetic as syn
    rng = np.random.default_rng(9)
    samples = syn.make_samples(100000)
    Q, S = 12, 100000
    ll = -0.5 * rng.standard_normal((Q, S)) ** 2 * rng.uniform(2, 400, (Q, 1)) - 3.0 * rng.random((Q, 1))
    ll[0, ::7] = np.nan
    ll[1, ::3] = -np.inf
    ll[2] = np.nan
    zlo = rng.uniform(2.0, 3.0, Q)
    zhi = zlo + rng.uniform(0.2, 1.5, Q)
    zhi[3] = zlo[3]
    qs = (0.025, 0.16, 0.5, 0.84, 0.975)
    got = api.dla_posteriors(dict(sample_log_likelihoods_dla=ll, min_z_dlas=zlo, max_z_dlas=zhi), samples, qs)
    amb = assert_matches_oracle(got, ll, zlo, zhi, samples["offset_samples"], samples["log_nhi_samples"], qs)
    assert np.all(np.isnan(got[2])) and np.all(np.isnan(got[3])) and np.all(np.isfinite(got[[0, 1, 4]]))
    print("S = 100 000: %d ambiguous quantiles" % amb)


@pytest.mark.gpu
def test_repeatable_host_equals_device_and_halves(processed):
    host, samples, proc, out = processed["host"], processed["samples"], processed["proc"], processed["out"]
    a = proc.posteriors_device(out).cpu().numpy()
    b = proc.posteriors_device(out).cpu().numpy()
    assert a.tobytes() == b.tobytes()
    assert api.dla_posteriors(host, samples).tobytes() == a.tobytes()
    Q = a.shape[0]
    half = {k: v[:Q // 2] for k, v in out.items()}
    rest = {k: v[Q // 2:].contiguous() for k, v in out.items()}
    both = np.concatenate([proc.posteriors_device(half).cpu().numpy(), proc.posteriors_device(rest).cpu().numpy()])
    assert both.tobytes() == a.tobytes()


# ---- multi-DLA
@pytest.fixture(scope="module")
def multi_processed():
    """process_multi_device outputs (J = 4) of 240 synthetic mean-flux spectra, some with two injected DLAs."""
    from gp_dla_detection_b200 import synthetic as syn
    model = syn.make_model()
    samples = syn.make_samples(10000, with_lls=True)
    spectra = syn.make_spectra(model, 240, seed=12, dla_fraction=0.4, meanflux=True, second_dla_fraction=0.4)
    proc = api.DLAProcessor(model, samples, syn.make_prior(), device=0)
    out = proc.process_multi_device(*_planes(spectra), max_dlas=4, return_samples=True)
    host = {k: v.cpu().numpy() for k, v in out.items()}
    yield dict(proc=proc, samples=samples, out=out, host=host)
    proc.close()


def assert_multi_matches_oracle(got, ll, part, zlo, zhi, off, lnhi, rtol=1e-12):
    Q, J, S = ll.shape
    ref = O.multi_dla_posteriors(ll, part, zlo, zhi, off, lnhi)
    assert got.shape == ref.shape
    assert np.array_equal(np.isnan(got), np.isnan(ref))
    g, r = api.unpack_multi_dla_posteriors(got, J), api.unpack_multi_dla_posteriors(ref, J)
    for n, floor in (("ess", None), ("z_mean", None), ("log_nhi_mean", None), ("z_sd", "z_mean"),
                     ("log_nhi_sd", "log_nhi_mean")):
        f = np.isfinite(r[n])
        fl = 0.0 if floor is None else 4e-16 * np.abs(r[floor][f])
        bad = ~_scaled_close(g[n][f], r[n][f], rtol, fl)
        assert not np.any(bad), (n, g[n][f][bad][:3], r[n][f][bad][:3])
    return r


@pytest.mark.gpu
def test_multi_kernel_matches_oracle_on_processed_quasars(multi_processed):
    host, samples, proc = multi_processed["host"], multi_processed["samples"], multi_processed["proc"]
    got = proc.multi_posteriors_device(multi_processed["out"]).cpu().numpy()
    r = assert_multi_matches_oracle(got, host["sample_log_likelihoods_dla"], host["base_sample_inds"],
                                    host["min_z_dlas"], host["max_z_dlas"], samples["offset_samples"],
                                    samples["log_nhi_samples"])
    per_level = np.count_nonzero(np.isfinite(r["ess"]), axis=0)
    print("multi-DLA: finite records per level 1..4: %s of %d" % (per_level.tolist(), got.shape[0]))
    assert per_level[0] > 0.9 * got.shape[0]
    # a level the run never reached (its row all NaN) is NaN
    unreached = np.all(np.isnan(host["sample_log_likelihoods_dla"]), axis=2)
    assert np.all(np.isnan(r["ess"][unreached]))
    # repeatable, and the host entry gives the same bits
    assert proc.multi_posteriors_device(multi_processed["out"]).cpu().numpy().tobytes() == got.tobytes()
    ref_layout = dict(host)
    ref_layout["sample_log_likelihoods_dla"] = np.transpose(host["sample_log_likelihoods_dla"], (0, 2, 1))
    ref_layout["base_sample_inds"] = np.transpose(host["base_sample_inds"], (0, 2, 1))
    assert api.multi_dla_posteriors(ref_layout, samples).tobytes() == got.tobytes()


@pytest.mark.gpu
def test_multi_one_level_matches_single_dla_kernel(multi_processed):
    proc, out = multi_processed["proc"], multi_processed["out"]
    one = dict(sample_log_likelihoods_dla=out["sample_log_likelihoods_dla"][:, :1].contiguous(),
               min_z_dlas=out["min_z_dlas"], max_z_dlas=out["max_z_dlas"])
    single = dict(sample_log_likelihoods_dla=out["sample_log_likelihoods_dla"][:, 0].contiguous(),
                  min_z_dlas=out["min_z_dlas"], max_z_dlas=out["max_z_dlas"])
    m = proc.multi_posteriors_device(one).cpu().numpy()
    s = proc.posteriors_device(single).cpu().numpy()[:, :5]
    assert np.array_equal(np.isnan(m), np.isnan(s))
    f = np.isfinite(s[:, 0])
    assert np.count_nonzero(f) > 100
    for c, floor in ((0, 0), (1, 0), (2, 4e-16 * np.abs(s[f, 1])), (3, 0), (4, 4e-16 * np.abs(s[f, 3]))):
        assert np.all(_scaled_close(m[f, c], s[f, c], 1e-12, floor)), c


@pytest.mark.gpu
def test_multi_unreached_level_and_poisoned_partner(multi_processed):
    import torch
    proc, out, samples = multi_processed["proc"], multi_processed["out"], multi_processed["samples"]
    J, S = 4, out["sample_log_likelihoods_dla"].shape[2]
    base = proc.multi_posteriors_device(out).cpu().numpy()
    ll = out["sample_log_likelihoods_dla"].clone()
    part = out["base_sample_inds"].clone()
    ll[3, 3] = float("nan")                                     # quasar 3 never reached level 4
    part[5, 1, 17] = S                                          # quasar 5: partner row 1 (levels 3, 4) out of range
    part[6, 0, 0] = -1                                          # quasar 6: partner row 0 (levels 2 to 4)
    mod = dict(out, sample_log_likelihoods_dla=ll, base_sample_inds=part)
    got = proc.multi_posteriors_device(mod).cpu().numpy()
    lev = lambda j: slice(j - 1 + 2 * (j - 1) * j, j + 2 * j * (j + 1))   # the columns of level j
    for q, nan_from in ((3, 4), (5, 3), (6, 2)):
        for j in range(1, J + 1):
            if j >= nan_from:
                assert np.all(np.isnan(got[q, lev(j)])), (q, j)
            else:
                assert got[q, lev(j)].tobytes() == base[q, lev(j)].tobytes(), (q, j)
    untouched = [q for q in range(base.shape[0]) if q not in (3, 5, 6)]
    assert got[untouched].tobytes() == base[untouched].tobytes()
    assert np.all(np.isfinite(base[[5, 6], :lev(2).stop]))       # the poisoned levels were finite before


# ---- calibration
def _sbc_spectra(model, samples, Q, num_lines, seed):
    """Spectra whose window flux is drawn from the inference model itself at a uniformly drawn sample (z, N)."""
    from gp_dla_detection_b200 import synthetic as syn
    from oracle import process_qsos_oracle as R
    rng = np.random.default_rng(seed)
    sp = syn.make_spectra(model, Q, seed=seed, dla_fraction=0.0)
    c_0, tau_0, beta = math.exp(model["log_c_0"]), math.exp(model["log_tau_0"]), math.exp(model["log_beta"])
    off, nhi = samples["offset_samples"], samples["nhi_samples"]
    truth = rng.integers(0, off.size, Q)
    for q in range(Q):
        wl, z_qso = sp["all_wavelengths"][q], float(sp["z_qsos"][q])
        mask, v = np.asarray(sp["all_pixel_mask"][q], bool), sp["all_noise_variance"][q]
        rest = wl / (1 + z_qso)
        window = (rest >= R.min_lambda) & (rest <= R.max_lambda)
        ind = window & ~mask
        lam = wl[ind]
        zlo, zhi = R.min_z_dla(lam, z_qso), R.max_z_dla(lam, z_qso)
        z_dla = zlo + (zhi - zlo) * off[truth[q]]
        a = R.voigt(R.padded_wavelengths(wl[window]), z_dla, nhi[truth[q]], num_lines)[~mask[window]]
        mu = np.interp(rest[ind], model["rest_wavelengths"], model["mu"])
        M = np.stack([np.interp(rest[ind], model["rest_wavelengths"], model["M"][:, j])
                      for j in range(model["M"].shape[1])], axis=1)
        om2 = np.exp(2.0 * np.interp(rest[ind], model["rest_wavelengths"], model["log_omega"]))
        om2 = om2 * (1.0 - np.exp(-tau_0 * (1.0 + (lam - R.lya_wavelength) / R.lya_wavelength) ** beta) + c_0) ** 2
        u, e1, e2 = rng.standard_normal(M.shape[1]), rng.standard_normal(lam.size), rng.standard_normal(lam.size)
        flux = np.array(sp["all_flux"][q], dtype=np.float64)
        flux[ind] = a * (mu + M @ u + np.sqrt(om2) * e1) + np.sqrt(v[ind]) * e2
        sp["all_flux"][q] = flux
    return sp, truth


def _coverage_check(truth_values, q_values, probs, w_max):
    """For each p: (count of truths <= q_p, lower bound, upper bound, inside)."""
    Q = truth_values.size
    rows = []
    for k, p in enumerate(probs):
        n = int(np.count_nonzero(truth_values <= q_values[:, k]))
        sigma = math.sqrt(Q * p * (1 - p))
        lo, hi = Q * p - 4 * sigma, Q * (p + np.mean(w_max)) + 4 * sigma
        rows.append((p, n, lo, hi, lo <= n <= hi))
    return rows


@pytest.mark.gpu
def test_simulation_based_calibration():
    """Truths drawn from the sample prior, flux from the inference model: P(truth <= q_p) lies in [p, p + w_max]."""
    from gp_dla_detection_b200 import synthetic as syn
    model = syn.make_model()
    samples = syn.make_samples(10000)
    Q, probs = 500, tuple(np.round(np.arange(1, 10) / 10.0, 1))
    proc = api.DLAProcessor(model, samples, syn.make_prior(), device=0)
    try:
        sp, truth = _sbc_spectra(model, samples, Q, proc.params.num_lines, seed=31)
        out = proc.process_device(*_planes(sp), return_sample_log_likelihoods=True)
        rec = proc.posteriors_device(out, quantiles=probs).cpu().numpy()
        ll = out["sample_log_likelihoods_dla"].cpu().numpy()
        zlo, zhi = out["min_z_dlas"].cpu().numpy(), out["max_z_dlas"].cpu().numpy()
    finally:
        proc.close()
    assert np.all(np.isfinite(rec))
    t = api.unpack_dla_posteriors(rec, len(probs))
    w = np.exp(ll - ll.max(axis=1, keepdims=True))
    w_max = 1.0 / w.sum(axis=1)
    z_true = zlo + (zhi - zlo) * samples["offset_samples"][truth]
    n_true = samples["log_nhi_samples"][truth]
    perm = np.random.default_rng(5).permutation(Q)
    print("SBC: ess percentiles 5/25/50/75/95 = %s; mean w_max = %.3f"
          % (np.array2string(np.percentile(t["ess"], [5, 25, 50, 75, 95]), precision=1), w_max.mean()))
    for name, truths, qv in (("z", z_true, t["z_quantiles"]), ("log N", n_true, t["log_nhi_quantiles"])):
        rows = _coverage_check(truths, qv, probs, w_max)
        control = _coverage_check(truths[perm], qv, probs, w_max)
        for (p, n, lo, hi, ok), (_, nc, _, _, okc) in zip(rows, control):
            print("SBC %-5s p = %.1f: %3d truths <= q_p, allowed [%.1f, %.1f]; permuted control %3d%s"
                  % (name, p, n, lo, hi, nc, "" if okc else " (outside)"))
        assert all(r[4] for r in rows), name
        assert not all(r[4] for r in control), name + ": the permuted control passes the check"


@pytest.mark.gpu
def test_end_to_end_intervals_on_injected_dlas():
    """Injection uses an unconvolved Ly-alpha-only profile, not the inference model: coverage is reported, not held
    to a bar."""
    from gp_dla_detection_b200 import synthetic as syn
    model = syn.make_model()
    samples = syn.make_samples(10000)
    spectra = syn.make_spectra(model, 2000, seed=21, dla_fraction=0.3)
    proc = api.DLAProcessor(model, samples, syn.make_prior(), device=0)
    try:
        out = proc.process_device(*_planes(spectra), return_sample_log_likelihoods=True)
        rec = proc.posteriors_device(out).cpu().numpy()
        p = out["p_dlas"].cpu().numpy()
        map_z, map_n = out["map_z_dlas"].cpu().numpy(), out["map_log_nhis"].cpu().numpy()
    finally:
        proc.close()
    t = api.unpack_dla_posteriors(rec, 5, num_samples=10000, p_dlas=p)
    fin = np.isfinite(p)
    assert np.all(np.isfinite(rec[fin]))
    for k in ("z_quantiles", "log_nhi_quantiles"):
        assert np.all(np.diff(t[k][fin], axis=1) >= 0), k
    det = fin & (p > 0.9)
    inside = ((map_z >= t["z_quantiles"][:, 0]) & (map_z <= t["z_quantiles"][:, 4])
              & (map_n >= t["log_nhi_quantiles"][:, 0]) & (map_n <= t["log_nhi_quantiles"][:, 4]))
    frac_map = np.count_nonzero(inside[det]) / max(np.count_nonzero(det), 1)
    inj = fin & np.isfinite(spectra["truth_log_nhi"])
    tn = spectra["truth_log_nhi"][inj]
    qn = t["log_nhi_quantiles"][inj]
    c68 = np.mean((tn >= qn[:, 1]) & (tn <= qn[:, 3]))
    c95 = np.mean((tn >= qn[:, 0]) & (tn <= qn[:, 4]))
    print("end-to-end: %d injected DLAs; truth log N inside the 68 %% interval %.3f, inside the 95 %% interval %.3f; "
          "mean p_dla_mc_sd %.2e; %d detections (p_dla > 0.9), MAP inside the 95 %% box for %.3f"
          % (inj.sum(), c68, c95, np.nanmean(t["p_dla_mc_sd"]), det.sum(), frac_map))
    assert det.sum() > 100 and frac_map >= 0.9
