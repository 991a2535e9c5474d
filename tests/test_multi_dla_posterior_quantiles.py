"""Credible intervals of every absorber of the multi-DLA model (per level and rank: the mass above the DLA threshold and
quantiles of z and log N): the NumPy restatement pinned on the CPU, the C entries' argument checks, the record layout,
the sharded gather, and on the GPU the kernel against the restatement, its determinism, NaN rules and both paths."""
import ctypes
import os
import socket

import numpy as np
import pytest

from gp_dla_detection_b200 import _lib, api
from gp_dla_detection_b200 import sharding as sh
from oracle import dla_posteriors_oracle as O
from oracle import multi_dla_posterior_quantiles_oracle as MQ


def _random_quasar(rng, S, J, scale=5.0):
    off, lnhi = rng.random(S), rng.uniform(20.0, 22.5, S)
    ll = -0.5 * rng.standard_normal((J, S)) ** 2 * scale
    part = rng.integers(0, S, (J - 1, S))
    return ll, part, off, lnhi


def reference(vals, w, ps, tol):
    """For each p: (the literal lower quantile, the sorted values a kernel may report at tolerance tol) from ONE stable
    sort; the same sets as O.acceptable_quantiles (pinned below), fast enough for thousands of rows."""
    order = np.argsort(vals, kind="stable")
    vs, c = vals[order], np.cumsum(w[order])
    out = []
    for p in ps:
        t, slack = p * c[-1], tol * c[-1]
        lo = int(np.searchsorted(c, t - slack, side="left"))
        hi = min(int(np.searchsorted(c, t + slack, side="left")), vs.size - 1)
        out.append((vs[int(np.searchsorted(c, t, side="left"))], np.unique(vs[lo:hi + 1])))
    return out


# ------------------------------------------------------------------ the restatement
def test_reference_sets_are_the_oracles():
    rng = np.random.default_rng(1)
    for S in (5, 64, 1000):
        vals = np.round(rng.random(S), 2)                        # ties in value
        w = np.exp(-0.5 * rng.standard_normal(S) ** 2 * 8)
        w[::5] = 0.0
        ps = (0.01, 0.3, 0.5, 0.97)
        for tol in (1e-12, 1e-3):
            for (lq, ok), p in zip(reference(vals, w, ps, tol), ps):
                assert lq == O.lower_quantile(vals, w, p)
                assert np.array_equal(ok, O.acceptable_quantiles(vals, w, p, tol)[0])


def test_one_level_is_the_single_dla_oracle():
    rng = np.random.default_rng(4)
    S, qs = 300, (0.025, 0.5, 0.9)
    off, lnhi = rng.random(S), rng.uniform(20.0, 22.5, S)
    ll = -0.5 * rng.standard_normal((6, 1, S)) ** 2 * 5
    ll[1, 0, ::3] = np.nan
    ll[2, 0] = -np.inf
    zlo, zhi = rng.uniform(2.0, 3.0, 6), rng.uniform(2.0, 4.0, 6)   # some empty ranges
    multi = MQ.multi_dla_posterior_quantiles(ll, None, zlo, zhi, off, lnhi, qs, threshold=21.0)
    single = O.dla_posteriors(ll[:, 0], zlo, zhi, off, lnhi, qs, threshold=21.0)
    assert multi.shape == (6, 7)
    assert np.array_equal(multi, single[:, 6:], equal_nan=True)     # mass, z quantiles, log-N quantiles
    assert np.any(np.isnan(multi[:, 0])) and np.any(np.isfinite(multi[:, 0]))


def test_every_partner_on_one_sample():
    """Level 2 with every partner at sample k: rank 0 is min(z_i, z_k) and rank 1 max(z_i, z_k), by hand."""
    off = np.array([0.1, 0.6, 0.3, 0.9, 0.05])                 # z = 2.1, 2.6, 2.3, 2.9, 2.05 in [2, 3]
    lnhi = np.array([20.0, 20.5, 21.5, 20.35, 19.5])
    ll = np.array([[0.0] * 5, [-np.inf, 0.0, 0.0, 0.0, -np.inf]])  # level 2: samples 1, 2, 3 with equal weight
    part = np.full((1, 5), 2)                                    # every partner: sample 2 (z 2.3, log N 21.5)
    rec = MQ.multi_quasar_posterior_quantiles(ll, part, 2.0, 3.0, off, lnhi, [0.3, 0.5, 0.9], threshold=21.0)
    t = api.unpack_multi_dla_posterior_quantiles(rec[None], 2, 3)
    z = lambda o: 2.0 + (3.0 - 2.0) * o
    # sample 1: (2.3, 2.6); sample 2: (2.3, 2.3), ties ranked by slot; sample 3: (2.3, 2.9)
    assert t["z_quantiles"][0, 1, 0].tolist() == [z(0.3)] * 3
    assert t["z_quantiles"][0, 1, 1].tolist() == [z(0.3), z(0.6), z(0.9)]
    # log N: sample 1 ranks (21.5, 20.5), sample 2 (21.5, 21.5), sample 3 (21.5, 20.35)
    assert t["log_nhi_quantiles"][0, 1, 0].tolist() == [21.5] * 3
    assert t["log_nhi_quantiles"][0, 1, 1].tolist() == [20.35, 20.5, 21.5]
    assert t["mass_above_threshold"][0, 1, 0] == 1.0 and abs(t["mass_above_threshold"][0, 1, 1] - 1 / 3) < 1e-16
    assert np.all(np.isnan(t["z_quantiles"][0, 0, 1]))           # rank 1 of level 1 does not exist


def test_ranks_are_stochastically_ordered():
    """The rank-r value is pointwise <= the rank-(r + 1) value, so every quantile is too."""
    rng = np.random.default_rng(5)
    S, J, qs = 400, 4, tuple(np.linspace(0.02, 0.98, 9))
    for trial in range(6):
        ll, part, off, lnhi = _random_quasar(rng, S, J, scale=rng.uniform(1, 30))
        rec = MQ.multi_quasar_posterior_quantiles(ll, part, 2.2, 3.4, off, lnhi, qs)
        t = api.unpack_multi_dla_posterior_quantiles(rec[None], J, len(qs))
        for j in range(2, J + 1):
            assert np.all(np.diff(t["z_quantiles"][0, j - 1, :j], axis=0) >= 0), (trial, j)
            assert np.all(np.diff(t["z_quantiles"][0, j - 1, :j], axis=1) >= 0), (trial, j)


def test_unpack_layout():
    J, P = 3, 2
    W = api.multi_dla_posterior_quantiles_width(J, P)
    assert W == 6 * 5 and api.multi_dla_posterior_quantiles_width(4, 5) == 110 == MQ.width(4, 5)
    rec = np.arange(2 * W, dtype=np.float64).reshape(2, W)
    t = api.unpack_multi_dla_posterior_quantiles(rec, J, P)
    assert t["mass_above_threshold"].shape == (2, J, J) and t["z_quantiles"].shape == (2, J, J, P)
    # level 1: [0..5), level 2: [5..15), level 3: [15..30); per rank: mass, z_q[P], log_nhi_q[P]
    assert t["mass_above_threshold"][1, 0, 0] == W and t["z_quantiles"][1, 0, 0].tolist() == [W + 1, W + 2]
    assert t["log_nhi_quantiles"][0, 1, 1].tolist() == [13.0, 14.0] and t["mass_above_threshold"][0, 2, 2] == 25.0
    assert np.all(np.isnan(t["mass_above_threshold"][:, 0, 1:])) and np.all(np.isnan(t["z_quantiles"][:, 1, 2]))
    with pytest.raises(ValueError):
        api.unpack_multi_dla_posterior_quantiles(rec, J, P + 1)


# ------------------------------------------------------------------ the C entries' argument checks (no GPU needed)
def _call(device=False, Q=1, S=4, max_dlas=3, quantiles=(0.5,), P=None, threshold=20.3, null=None):
    lib = _lib.load()
    J, n, s = min(max(max_dlas, 1), 4), min(max(Q, 1), 4), max(S, 1)
    qs = np.asarray(quantiles, dtype=np.float64)
    ll, part = np.zeros((n, J, s)), np.zeros((n, max(J - 1, 1), s), dtype=np.int32)
    zlo, zhi, off, lnhi = np.full(n, 2.0), np.full(n, 3.0), np.linspace(0, 1, s), np.full(s, 21.0)
    out = np.zeros((n, MQ.width(J, max(qs.size, 1))))
    vp = lambda a, k: None if null == k else ctypes.c_void_p(a.ctypes.data)
    args = [Q, S, max_dlas, vp(ll, "ll"), vp(part, "part"), vp(zlo, "zlo"), vp(zhi, "zhi"), vp(off, "off"),
            vp(lnhi, "lnhi"), qs.size if P is None else P, None if null == "quantiles" else api._dp(qs), threshold,
            vp(out, "out")]
    if device:
        rc = lib.gpdla_multi_dla_posterior_quantiles_device(*args, None)
    else:
        rc = lib.gpdla_multi_dla_posterior_quantiles(*args)
    return rc, (lib.gpdla_last_error(None) or b"").decode()


BAD = dict(max_dlas_zero=dict(max_dlas=0), max_dlas_five=dict(max_dlas=5), null_partners=dict(null="part"),
           null_ll=dict(null="ll"), null_log_nhi=dict(null="lnhi"), zero_s=dict(S=0), negative_q=dict(Q=-1),
           big_q=dict(Q=2 ** 31), null_out=dict(null="out"), null_zlo=dict(null="zlo"),
           no_quantiles=dict(quantiles=(), P=0), seventeen=dict(quantiles=np.full(17, 0.5)),
           p_zero=dict(quantiles=(0.0, 0.5)), p_one=dict(quantiles=(0.5, 1.0)), p_nan=dict(quantiles=(np.nan,)),
           p_negative=dict(quantiles=(-0.1,)), threshold_nan=dict(threshold=np.nan),
           threshold_inf=dict(threshold=-np.inf), null_quantiles=dict(null="quantiles"))


@pytest.mark.parametrize("device", [False, True])
@pytest.mark.parametrize("case", sorted(BAD))
def test_c_entries_reject_bad_arguments(case, device):
    rc, msg = _call(device=device, **BAD[case])
    assert rc == _lib.GPDLA_ERR_INVALID, (rc, msg)
    name = "gpdla_multi_dla_posterior_quantiles" + ("_device" if device else "")
    assert msg.startswith(name + ": "), msg


def test_c_entries_accept_the_limits():
    """1 and 16 quantiles, 1 level without partners and 4 levels, and Q = 0 pass the checks (a non-empty call then
    needs a device)."""
    import torch
    want = _lib.GPDLA_OK if torch.cuda.is_available() else _lib.GPDLA_ERR_CUDA
    for kw in (dict(quantiles=(0.5,)), dict(quantiles=np.linspace(0.01, 0.99, 16)), dict(max_dlas=1, null="part"),
               dict(max_dlas=4, quantiles=(0.1, 0.9))):
        rc, msg = _call(**kw)
        assert rc == want, (kw, msg)
    rc, msg = _call(device=True, Q=0, null="ll")
    assert rc == _lib.GPDLA_OK, msg


# ------------------------------------------------------------------ sharded gather, 2 gloo ranks, CPU stand-in
S_STAND_IN, J_STAND_IN, QUANTILES = 64, 2, (0.1, 0.5, 0.9)


def _stand_in_records(sp):
    """Oracle records of deterministic stand-ins for process_multi_device outputs, keyed on z_qso."""
    z = np.asarray(sp["z_qsos"])
    S = S_STAND_IN
    off, lnhi = (np.arange(S) + 0.5) / S, 20.0 + 3.0 * ((np.arange(S) * 0.618034) % 1.0)
    c = np.modf(7.0 * z)[0]
    ll = -50.0 * (off[None, None, :] - c[:, None, None] * np.array([1.0, 0.5])[None, :, None]) ** 2
    part = ((np.arange(S)[None, None, :] * 5 + np.round(c * S).astype(int)[:, None, None]) % S)
    zlo, zhi = z - 1.0, z - 0.05
    return (O.multi_dla_posteriors(ll, part, zlo, zhi, off, lnhi),
            MQ.multi_dla_posterior_quantiles(ll, part, zlo, zhi, off, lnhi, QUANTILES))


def _sharded_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from gp_dla_detection_b200 import synthetic as syn
    spectra = syn.make_spectra(syn.make_model(), 11, seed=6)
    res = sh.multi_dla_posteriors_sharded(None, None, spectra, None, quantiles=QUANTILES, max_dlas=J_STAND_IN,
                                          batch_quasars=2, compute=_stand_in_records)
    q.put((rank, res["records"].tobytes(), res["quantile_records"].tobytes(), res["quantile_records"].shape,
           res["blocks"]))
    dist.destroy_process_group()


def test_sharded_multi_posteriors_two_gloo_ranks():
    import torch.multiprocessing as mp
    from gp_dla_detection_b200 import synthetic as syn
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_sharded_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    results = sorted(q.get(timeout=180) for _ in range(2))
    for p in procs:
        p.join(60)
    (r0, m0, q0, shape, blocks), (r1, m1, q1, _, _) = results
    assert (r0, r1) == (0, 1) and m0 == m1 and q0 == q1
    assert blocks[0][1] > 0 and blocks[1][1] > blocks[0][1]       # both ranks hold quasars
    ref_m, ref_q = _stand_in_records(syn.make_spectra(syn.make_model(), 11, seed=6))
    assert shape == (11, api.multi_dla_posterior_quantiles_width(J_STAND_IN, len(QUANTILES)))
    assert np.frombuffer(m0, dtype=np.float64).tobytes() == ref_m.tobytes()      # catalogue order, every bit
    assert np.frombuffer(q0, dtype=np.float64).tobytes() == ref_q.tobytes()
    assert np.all(np.isfinite(ref_q))


# ------------------------------------------------------------------ on the GPU
def _up(a, dt):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, dtype=dt)).cuda()


def _planes(spectra):
    pad = api.pad_spectra(spectra)
    return (_up(pad["wavelengths"], np.float64), _up(pad["flux"], np.float64), _up(pad["noise_variance"], np.float64),
            _up(pad["pixel_mask"], np.uint8), _up(pad["lengths"], np.int32), _up(pad["z_qsos"], np.float64))


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


def assert_matches_oracle(got, ll, part, zlo, zhi, off, lnhi, qs, thr=20.3, literal=24):
    """The NaN pattern of the restatement; the mass to 1e-12; every quantile in the set the restatement's cumulative
    sums allow at quantile_tolerance(S), and equal to its literal value where that set holds one value.  The first
    `literal` quasars are also compared with the literal restatement.  Returns (ambiguous, checked) counts."""
    Q, J, S = ll.shape
    P, tol = len(qs), MQ.quantile_tolerance(S)
    part = np.zeros((Q, 0, S), dtype=np.int64) if part is None else part
    lit = MQ.multi_dla_posterior_quantiles(ll[:literal], part[:literal], zlo[:literal], zhi[:literal], off, lnhi, qs,
                                           thr)
    g = api.unpack_multi_dla_posterior_quantiles(got, J, P)
    ref = np.full_like(got, np.nan)
    ambiguous = checked = 0
    for q in range(Q):
        c = 0
        for j in range(1, J + 1):
            w = O.weights(ll[q, j - 1])
            rows = part[q, :j - 1]
            if w is None or not zhi[q] > zlo[q] or np.any((rows < 0) | (rows >= S)):
                c += j * (1 + 2 * P)
                continue
            z, n = O.ranked_slots(part[q], j, zlo[q], zhi[q], off, lnhi)
            for r in range(j):
                ref[q, c] = np.sum(w[n[r] >= thr]) / np.sum(w)
                for base, vals, name in ((c + 1, z[r], "z_quantiles"), (c + 1 + P, n[r], "log_nhi_quantiles")):
                    for k, (lq, ok) in enumerate(reference(vals, w, qs, tol)):
                        ref[q, base + k] = lq
                        v = g[name][q, j - 1, r, k]
                        assert v in ok, (q, j, r, name, qs[k], v, ok, lq)
                        ambiguous += ok.size > 1
                        checked += 1
                        if ok.size == 1:
                            assert v == lq, (q, j, r, name, qs[k], v, lq)
                c += 1 + 2 * P
    assert np.array_equal(lit, ref[:literal], equal_nan=True)    # the fast restatement is the literal one
    assert np.array_equal(np.isnan(got), np.isnan(ref))
    f = np.isfinite(g["mass_above_threshold"])
    rm = api.unpack_multi_dla_posterior_quantiles(ref, J, P)["mass_above_threshold"]
    assert np.all(np.abs(g["mass_above_threshold"][f] - rm[f]) <= 1e-12), "mass_above_threshold"
    return ambiguous, checked


@pytest.mark.gpu
@pytest.mark.parametrize("P", [1, 5, 16])
def test_kernel_matches_oracle_on_processed_quasars(multi_processed, P):
    rng = np.random.default_rng(P)
    host, samples, proc = multi_processed["host"], multi_processed["samples"], multi_processed["proc"]
    qs = (0.5,) if P == 1 else api.DEFAULT_QUANTILES if P == 5 else tuple(rng.uniform(0.005, 0.995, P))
    thr = 20.3 if P != 16 else float(samples["log_nhi_samples"][123])   # a threshold on a stored sample value
    got = proc.multi_posterior_quantiles_device(multi_processed["out"], quantiles=qs, log_nhi_threshold=thr)
    got = got.cpu().numpy()
    amb, n = assert_matches_oracle(got, host["sample_log_likelihoods_dla"], host["base_sample_inds"],
                                   host["min_z_dlas"], host["max_z_dlas"], samples["offset_samples"],
                                   samples["log_nhi_samples"], qs, thr)
    per_level = [int(np.count_nonzero(np.isfinite(got[:, (j - 1) * j // 2 * (1 + 2 * P)]))) for j in range(1, 5)]
    print("P = %d: finite levels 1..4 %s of %d quasars; %d of %d quantiles had more than one acceptable value"
          % (P, per_level, got.shape[0], amb, n))
    assert per_level[0] > 0.9 * got.shape[0] and per_level[1] > 0


@pytest.mark.gpu
def test_repeatable_host_equals_device_and_halves(multi_processed):
    host, samples, proc, out = (multi_processed[k] for k in ("host", "samples", "proc", "out"))
    a = proc.multi_posterior_quantiles_device(out).cpu().numpy()
    assert proc.multi_posterior_quantiles_device(out).cpu().numpy().tobytes() == a.tobytes()
    ref_layout = dict(host)
    ref_layout["sample_log_likelihoods_dla"] = np.transpose(host["sample_log_likelihoods_dla"], (0, 2, 1))
    ref_layout["base_sample_inds"] = np.transpose(host["base_sample_inds"], (0, 2, 1))
    assert api.multi_dla_posterior_quantiles(ref_layout, samples).tobytes() == a.tobytes()
    Q = a.shape[0]
    half = {k: v[:Q // 2] for k, v in out.items()}
    rest = {k: v[Q // 2:].contiguous() for k, v in out.items()}
    both = np.concatenate([proc.multi_posterior_quantiles_device(half).cpu().numpy(),
                           proc.multi_posterior_quantiles_device(rest).cpu().numpy()])
    assert both.tobytes() == a.tobytes()


@pytest.mark.gpu
def test_one_level_matches_single_dla_kernel(multi_processed):
    proc, out, samples = multi_processed["proc"], multi_processed["out"], multi_processed["samples"]
    qs = api.DEFAULT_QUANTILES
    P = len(qs)
    one = dict(sample_log_likelihoods_dla=out["sample_log_likelihoods_dla"][:, :1].contiguous(),
               min_z_dlas=out["min_z_dlas"], max_z_dlas=out["max_z_dlas"])
    single = dict(sample_log_likelihoods_dla=out["sample_log_likelihoods_dla"][:, 0].contiguous(),
                  min_z_dlas=out["min_z_dlas"], max_z_dlas=out["max_z_dlas"])
    m = proc.multi_posterior_quantiles_device(one, qs).cpu().numpy()
    s = proc.posteriors_device(single, qs).cpu().numpy()[:, 6:]
    assert m.shape == s.shape and np.array_equal(np.isnan(m), np.isnan(s))
    f = np.isfinite(s[:, 0])
    assert np.count_nonzero(f) > 100
    assert np.all(np.abs(m[f, 0] - s[f, 0]) <= 1e-12)
    ll, zlo, zhi = (multi_processed["host"][k] for k in ("sample_log_likelihoods_dla", "min_z_dlas", "max_z_dlas"))
    off, lnhi = samples["offset_samples"], samples["log_nhi_samples"]
    tol = MQ.quantile_tolerance(off.size)
    for q in np.flatnonzero(f):
        w = O.weights(ll[q, 0])
        for base, vals in ((1, O.sample_z(zlo[q], zhi[q], off)), (1 + P, lnhi)):
            for k, (_, ok) in enumerate(reference(vals, w, qs, tol)):
                assert m[q, base + k] in ok and s[q, base + k] in ok, (q, base + k)


@pytest.mark.gpu
def test_unreached_level_and_poisoned_partners(multi_processed):
    proc, out = multi_processed["proc"], multi_processed["out"]
    J, S, P = 4, out["sample_log_likelihoods_dla"].shape[2], 5
    base = proc.multi_posterior_quantiles_device(out).cpu().numpy()
    ll = out["sample_log_likelihoods_dla"].clone()
    part = out["base_sample_inds"].clone()
    ll[3, 3] = float("nan")                                     # quasar 3 never reached level 4
    part[5, 1, 17] = S                                          # quasar 5: partner row 1 (levels 3, 4) out of range
    part[6, 0, 0] = -1                                          # quasar 6: partner row 0 (levels 2 to 4)
    mod = dict(out, sample_log_likelihoods_dla=ll, base_sample_inds=part)
    got = proc.multi_posterior_quantiles_device(mod).cpu().numpy()
    moments = proc.multi_posteriors_device(mod).cpu().numpy()
    lev = lambda j: slice((j - 1) * j // 2 * (1 + 2 * P), j * (j + 1) // 2 * (1 + 2 * P))
    mlev = lambda j: slice(j - 1 + 2 * (j - 1) * j, j + 2 * j * (j + 1))
    for q in range(got.shape[0]):
        for j in range(1, J + 1):
            if np.isnan(moments[q, mlev(j)][0]):                # NaN exactly where the moments kernel gives NaN
                assert np.all(np.isnan(got[q, lev(j)])), (q, j)
            else:                                               # and every other level keeps its bits
                assert got[q, lev(j)].tobytes() == base[q, lev(j)].tobytes(), (q, j)
    for q, nan_from in ((3, 4), (5, 3), (6, 2)):
        assert np.all(np.isnan(got[q, lev(nan_from).start:])), q
    assert np.all(np.isfinite(base[[5, 6], :lev(2).stop]))       # the poisoned levels were finite before


def _synthetic_rows(rng, Q, J, S, crowded=()):
    ll = -0.5 * rng.standard_normal((Q, J, S)) ** 2 * rng.uniform(2, 400, (Q, J, 1)) - 3.0 * rng.random((Q, J, 1))
    part = rng.integers(0, S, (Q, J - 1, S)).astype(np.int32)
    for q in crowded:                                           # every partner on one sample: one bin takes them all
        part[q] = rng.integers(0, S)
    zlo = rng.uniform(2.0, 3.0, Q)
    return ll, part, zlo, zlo + rng.uniform(0.2, 1.5, Q)


def _host_layout(ll, part, zlo, zhi):
    return dict(sample_log_likelihoods_dla=np.transpose(ll, (0, 2, 1)), base_sample_inds=np.transpose(part, (0, 2, 1)),
                min_z_dlas=zlo, max_z_dlas=zhi)


@pytest.mark.gpu
def test_large_sample_count_global_scratch():
    """S = 100 000: the histograms live in each resident CTA's global scratch; one quasar has crowded partners."""
    from gp_dla_detection_b200 import synthetic as syn
    rng = np.random.default_rng(9)
    Q, J, S = 6, 3, 100000
    samples = syn.make_samples(S)
    ll, part, zlo, zhi = _synthetic_rows(rng, Q, J, S, crowded=(1,))
    ll[0, 1, ::3] = -np.inf
    ll[2, 2] = np.nan
    zhi[3] = zlo[3]
    qs = api.DEFAULT_QUANTILES
    got = api.multi_dla_posterior_quantiles(_host_layout(ll, part, zlo, zhi), samples, qs)
    amb, n = assert_matches_oracle(got, ll, part, zlo, zhi, samples["offset_samples"], samples["log_nhi_samples"], qs,
                                   literal=2)
    assert np.all(np.isnan(got[3])) and np.all(np.isfinite(got[[0, 1, 4, 5]]))
    print("S = 100 000: %d of %d quantiles had more than one acceptable value" % (amb, n))


@pytest.mark.gpu
def test_crowded_partners_in_shared_memory():
    """Every partner of a quasar on one sample: whole warps add into one bin."""
    from gp_dla_detection_b200 import synthetic as syn
    rng = np.random.default_rng(10)
    Q, J, S = 8, 4, 10000
    samples = syn.make_samples(S)
    ll, part, zlo, zhi = _synthetic_rows(rng, Q, J, S, crowded=range(Q))
    ll[:4] = -1e-3 * rng.random((4, J, S))                       # near-flat weights: every sample counts
    qs = (0.01, 0.16, 0.5, 0.84, 0.99)
    got = api.multi_dla_posterior_quantiles(_host_layout(ll, part, zlo, zhi), samples, qs)
    amb, n = assert_matches_oracle(got, ll, part, zlo, zhi, samples["offset_samples"], samples["log_nhi_samples"], qs,
                                   literal=3)
    assert np.all(np.isfinite(got))
    print("crowded partners: %d of %d quantiles had more than one acceptable value" % (amb, n))


@pytest.mark.gpu
def test_end_to_end_intervals_on_two_dla_spectra():
    """Injection uses an unconvolved Ly-alpha-only profile, not the inference model: coverage is reported, not held
    to a bar."""
    from gp_dla_detection_b200 import synthetic as syn
    model = syn.make_model()
    samples = syn.make_samples(10000, with_lls=True)
    spectra = syn.make_spectra(model, 2000, seed=22, dla_fraction=0.4, meanflux=True, second_dla_fraction=0.5)
    proc = api.DLAProcessor(model, samples, syn.make_prior(), device=0)
    try:
        out = proc.process_multi_device(*_planes(spectra), max_dlas=4, return_samples=True)
        rec = proc.multi_posterior_quantiles_device(out).cpu().numpy()
    finally:
        proc.close()
    t = api.unpack_multi_dla_posterior_quantiles(rec, 4, 5)
    two = np.isfinite(spectra["truth_z_dla"]) & np.isfinite(spectra["truth_z_dla2"])
    two &= np.all(np.isfinite(t["z_quantiles"][:, 1, :2]), axis=(1, 2))
    assert two.sum() > 50
    tz = np.sort(np.stack([spectra["truth_z_dla"], spectra["truth_z_dla2"]], axis=1), axis=1)[two]
    first = spectra["truth_z_dla"] <= spectra["truth_z_dla2"]
    tn = np.where(first[:, None], np.stack([spectra["truth_log_nhi"], spectra["truth_log_nhi2"]], axis=1),
                  np.stack([spectra["truth_log_nhi2"], spectra["truth_log_nhi"]], axis=1))[two]
    zq, nq = t["z_quantiles"][two, 1, :2], t["log_nhi_quantiles"][two, 1, :2]   # level 2, ranks 0 and 1
    cover = lambda x, qv, a, b: np.mean((x >= qv[..., a]) & (x <= qv[..., b]))
    print("end-to-end: %d spectra with two injected DLAs; level-2 z inside 68 %% / 95 %% intervals %.3f / %.3f, "
          "log N %.3f / %.3f; mean level-2 DLA mass of the two ranks %s"
          % (two.sum(), cover(tz, zq, 1, 3), cover(tz, zq, 0, 4), cover(tn, nq, 1, 3), cover(tn, nq, 0, 4),
             np.array2string(np.mean(t["mass_above_threshold"][two, 1, :2], axis=0), precision=3)))
    assert np.all(np.diff(t["z_quantiles"][two, 1, :2], axis=2) >= 0)
