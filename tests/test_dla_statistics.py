"""Population statistics of the single-DLA catalogue (column density distribution, dN/dX, Omega_DLA): the NumPy
restatement pinned by hand values and exact enumerations on the CPU, the C entry's argument checks, the sharded sum,
and on the GPU the statistics kernel against the restatement."""
import ctypes
import itertools
import math
import os
import socket

import numpy as np
import pytest

from gp_dla_detection_b200 import _lib, api
from gp_dla_detection_b200 import sharding as sh
from oracle import dla_statistics_oracle as O


# ------------------------------------------------------------------ the restatement, by hand
def _hand_quasar():
    ll = np.log([1.0, 2.0, 3.0, 4.0, 10.0])                    # w = 0.05, 0.1, 0.15, 0.2, 0.5
    offset = np.array([0.1, 0.6, 0.3, 0.9, 0.05])              # z = 2.1, 2.6, 2.3, 2.9, 2.05 for z in [2, 3]
    log_nhi = np.array([20.0, 20.5, 21.5, 20.35, 19.5])
    return ll, offset, log_nhi, 10.0 ** log_nhi


def test_oracle_known_answer_one_quasar():
    ll, off, lnhi, nhi = _hand_quasar()
    p = 0.8
    z_edges, n_edges = [2.0, 2.5, 3.0], [20.0, 20.4, 21.0, 22.0]
    q, d, e, e2 = O.quasar_cells(ll, p, 2.0, 3.0, off, lnhi, nhi, z_edges, n_edges)
    w = np.array([1, 2, 3, 4, 10]) / 20.0
    q_ref = np.zeros((2, 3))
    q_ref[0, 0] = p * w[0]              # z 2.1, log N 20.0: not a DLA
    q_ref[1, 1] = p * w[1]              # z 2.6, 20.5
    q_ref[0, 2] = p * w[2]              # z 2.3, 21.5
    q_ref[1, 0] = p * w[3]              # z 2.9, 20.35 (>= 20.3: a DLA in the first log-N bin)
    # sample 4 (z 2.05, log N 19.5) is below every log-N bin and below the threshold: its weight counts nowhere
    np.testing.assert_allclose(q, q_ref, rtol=1e-15, atol=0)
    np.testing.assert_allclose(d, [p * w[2], p * (w[1] + w[3])], rtol=1e-15)
    np.testing.assert_allclose(e, [p * w[2] * nhi[2], p * (w[1] * nhi[1] + w[3] * nhi[3])], rtol=1e-15)
    np.testing.assert_allclose(e2, [p * w[2] * nhi[2] ** 2, p * (w[1] * nhi[1] ** 2 + w[3] * nhi[3] ** 2)], rtol=1e-15)
    sums = O.dla_statistics_sums(ll[None], [p], [2.0], [3.0], off, lnhi, nhi, z_edges, n_edges)
    t = api.unpack_dla_statistics(sums, 2, 3)
    np.testing.assert_allclose(t["counts_var"], q_ref * (1 - q_ref), rtol=1e-15)
    np.testing.assert_allclose(t["nhi_var"], e2 - e * e, rtol=1e-15)
    np.testing.assert_allclose(t["path"], [O.path_length(2, 3, 2, 2.5, 0.3), O.path_length(2, 3, 2.5, 3, 0.3)],
                               rtol=1e-15)
    assert t["num_quasars"] == 1.0


@pytest.mark.parametrize("why", ["nan_p", "select", "empty_z"])
def test_oracle_excluded_quasar_contributes_nothing(why):
    ll, off, lnhi, nhi = _hand_quasar()
    p, zlo, zhi, sel = [0.8], [2.0], [3.0], None
    if why == "nan_p":
        p = [np.nan]
    elif why == "select":
        sel = [False]
    else:
        zhi = [2.0]
    sums = O.dla_statistics_sums(ll[None], p, zlo, zhi, off, lnhi, nhi, [2.0, 2.5, 3.0], [20.0, 21.0], select=sel)
    assert np.array_equal(sums, np.zeros(api.dla_statistics_width(2, 1)))


def test_absorption_distance_against_quadrature():
    from scipy.integrate import quad
    for om in (0.3, 0.2726, 1.0):
        E = lambda z: math.sqrt(om * (1 + z) ** 3 + 1 - om)
        for z1, z2 in ((2.0, 2.5), (2.15, 5.1), (0.0, 1e-3)):
            ref = quad(lambda z: (1 + z) ** 2 / E(z), z1, z2, epsabs=0, epsrel=1e-13)[0]
            got = O.absorption_distance(z2, om) - O.absorption_distance(z1, om)
            assert abs(got - ref) <= 1e-10 * ref, (om, z1, z2)
    # clipped to [min_z, max_z] and the bin
    X = lambda z: float(O.absorption_distance(z, 0.3))
    assert O.path_length(2.2, 2.8, 2.0, 2.5, 0.3) == X(2.5) - X(2.2)
    assert O.path_length(2.2, 2.8, 2.5, 3.0, 0.3) == X(2.8) - X(2.5)
    assert O.path_length(2.2, 2.4, 2.5, 3.0, 0.3) == 0.0
    assert O.path_length(2.6, 2.8, 2.0, 2.5, 0.3) == 0.0


def test_count_variance_is_exact_poisson_binomial():
    rng = np.random.default_rng(3)
    for Q in (1, 5, 12):
        q = rng.random(Q) * rng.random(Q)
        mean = var = 0.0
        moments = np.zeros(3)
        for outcome in itertools.product((0, 1), repeat=Q):
            o = np.array(outcome)
            prob = np.prod(np.where(o == 1, q, 1 - q))
            n = o.sum()
            moments += prob * np.array([1.0, n, n * n])
        mean = moments[1]
        var = moments[2] - mean ** 2
        assert abs(moments[0] - 1) < 1e-12
        assert abs(mean - q.sum()) < 1e-12
        assert abs(var - np.sum(q * (1 - q))) < 1e-12


def test_nhi_variance_is_the_categorical_mixture():
    ll, off, lnhi, nhi = _hand_quasar()
    p = 0.7
    q, d, e, e2 = O.quasar_cells(ll, p, 2.0, 3.0, off, lnhi, nhi, [2.0, 3.0], [20.0, 22.0])
    # one quasar: with probability p w_j its DLA is sample j; its N_HI sum is N_j for a DLA sample in the bin, else 0
    w = np.exp(ll - ll.max()); w /= w.sum()
    x = np.where(lnhi >= 20.3, nhi, 0.0)
    mean = np.sum(p * w * x)
    var = np.sum(p * w * x * x) - mean ** 2
    assert abs(e[0] - mean) <= 1e-15 * mean
    assert abs((e2[0] - e[0] ** 2) - var) <= 1e-12 * var


def test_finish_formulas_and_units():
    assert abs(api.omega_dla_coefficient(0.7) - 1.375931e-23) < 1e-29
    assert api.omega_dla_coefficient(0.7) == O.omega_coefficient(0.7)
    z_edges, n_edges = [2.0, 3.0, 4.0], [20.0, 21.0, 22.0]
    rng = np.random.default_rng(1)
    sums = rng.random(api.dla_statistics_width(2, 2)) + 0.5
    got = api.finish_dla_statistics(sums, z_edges, n_edges, hubble_h=0.7)
    ref = O.finish(sums, z_edges, n_edges, hubble_h=0.7)
    for k, v in ref.items():
        np.testing.assert_allclose(got[k], v, rtol=1e-14, err_msg=k)
    # f(N) is per unit N_HI per unit X: one expected DLA in [20, 21) over unit path is 1 / (10^21 - 10^20)
    s = np.zeros(api.dla_statistics_width(1, 1))
    s[0] = 1.0
    s[2 + 4] = 1.0                                    # path of the single z bin
    f = api.finish_dla_statistics(s, [2.0, 3.0], [20.0, 21.0])
    assert f["cddf"][0, 0] == 1.0 / (1e21 - 1e20)
    assert f["dndx"][0] == 0.0 and f["path_length"][0] == 1.0


# ------------------------------------------------------------------ the C entry's argument checks (no GPU needed)
def _call_host(z_edges, n_edges, omega_m=0.3, Q=1, S=4):
    lib = _lib.load()
    ll, p, zlo, zhi = np.zeros((Q, S)), np.full(Q, 0.5), np.full(Q, 2.0), np.full(Q, 3.0)
    off, lnhi, nhi = np.linspace(0, 1, S), np.full(S, 21.0), np.full(S, 1e21)
    ze, ne = np.asarray(z_edges, float), np.asarray(n_edges, float)
    sums = np.zeros(max(api.dla_statistics_width(max(ze.size - 1, 0), max(ne.size - 1, 0)), 1))
    vp = lambda a: ctypes.c_void_p(a.ctypes.data)
    rc = lib.gpdla_dla_statistics(Q, S, vp(ll), vp(p), vp(zlo), vp(zhi), None, vp(off), vp(lnhi), vp(nhi), ze.size - 1,
                                  api._dp(ze), ne.size - 1, api._dp(ne), 20.3, omega_m, vp(sums))
    return rc, (lib.gpdla_last_error(None) or b"").decode()


@pytest.mark.parametrize("case", ["unsorted_z", "repeated_nhi", "nan_z", "inf_nhi", "too_many_z", "too_many_nhi",
                                  "omega_zero", "omega_negative", "omega_above_one"])
def test_c_entry_rejects_bad_arguments(case):
    z, n, om = [2.0, 2.5, 3.0], [20.0, 21.0, 22.0], 0.3
    if case == "unsorted_z":
        z = [2.0, 3.0, 2.5]
    elif case == "repeated_nhi":
        n = [20.0, 21.0, 21.0]
    elif case == "nan_z":
        z = [2.0, np.nan, 3.0]
    elif case == "inf_nhi":
        n = [20.0, 21.0, np.inf]
    elif case == "too_many_z":
        z = np.linspace(2.0, 3.0, 66)                 # 65 bins
    elif case == "too_many_nhi":
        n = np.linspace(20.0, 23.0, 130)              # 129 bins
    elif case == "omega_zero":
        om = 0.0
    elif case == "omega_negative":
        om = -0.3
    else:
        om = 1.5
    rc, msg = _call_host(z, n, om)
    assert rc == _lib.GPDLA_ERR_INVALID, (rc, msg)
    assert msg.startswith("gpdla_dla_statistics: "), msg


def test_c_entry_accepts_the_limits():
    """64 z bins and 128 log-N bins pass the checks (the call then needs a device)."""
    import torch
    rc, msg = _call_host(np.linspace(2.0, 3.0, 65), np.linspace(20.0, 23.0, 129), 1.0)
    assert rc == (_lib.GPDLA_OK if torch.cuda.is_available() else _lib.GPDLA_ERR_CUDA), msg


# ------------------------------------------------------------------ sharded sum, 2 gloo ranks, CPU stand-in
Z_EDGES, N_EDGES = [2.0, 2.6, 3.4, 6.0], [20.0, 20.5, 21.0, 22.0, 23.0]


def _stand_in_results(sp, S=64):
    """Deterministic per-quasar stand-ins for process_device outputs, keyed on z_qso."""
    z = np.asarray(sp["z_qsos"])
    off = (np.arange(S) + 0.5) / S
    ll = -50.0 * (off[None, :] - np.modf(7.0 * z)[0][:, None]) ** 2
    return ll, np.clip(z - 2.1, 0, 1), z - 1.0, z - 0.05


def _stand_in_samples(S=64):
    lnhi = 20.0 + 3.0 * ((np.arange(S) * 0.618034) % 1.0)
    return (np.arange(S) + 0.5) / S, lnhi, 10.0 ** lnhi


def _stats_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from gp_dla_detection_b200 import synthetic as syn
    model = syn.make_model()
    spectra = syn.make_spectra(model, 11, seed=6)
    select = np.arange(11) % 4 != 1
    off, lnhi, nhi = _stand_in_samples()

    def compute(sp, sel, sums):
        ll, p, zlo, zhi = _stand_in_results(sp)
        return O.dla_statistics_sums(ll, p, zlo, zhi, off, lnhi, nhi, Z_EDGES, N_EDGES, select=sel, sums=sums)
    res = sh.dla_statistics_sharded(model, None, spectra, None, Z_EDGES, N_EDGES, select=select, batch_quasars=2,
                                    compute=compute)
    q.put((rank, res["sums"].tobytes(), res["blocks"]))
    dist.destroy_process_group()


def test_sharded_statistics_two_gloo_ranks():
    import torch.multiprocessing as mp
    from gp_dla_detection_b200 import synthetic as syn
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_stats_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    results = sorted(q.get(timeout=180) for _ in range(2))
    for p in procs:
        p.join(60)
    (r0, b0, blocks), (r1, b1, _) = results
    assert (r0, r1) == (0, 1) and b0 == b1                     # every rank holds the same bits
    total = np.frombuffer(b0, dtype=np.float64)
    # the same sums in rank order, each rank's block in batches of 2
    spectra = syn.make_spectra(syn.make_model(), 11, seed=6)
    select = np.arange(11) % 4 != 1
    off, lnhi, nhi = _stand_in_samples()
    ranks = []
    for s0, e0 in blocks:
        acc = np.zeros(api.dla_statistics_width(3, 4))
        for a in range(s0, e0, 2):
            ll, p, zlo, zhi = _stand_in_results(sh.slice_spectra(spectra, a, min(e0, a + 2)))
            acc = O.dla_statistics_sums(ll, p, zlo, zhi, off, lnhi, nhi, Z_EDGES, N_EDGES, select=select[a:a + 2],
                                        sums=acc)
        ranks.append(acc)
    assert np.array_equal(total, ranks[0] + ranks[1])
    assert total[-1] == np.count_nonzero(select)               # the stand-in makes every selected quasar contribute


# ------------------------------------------------------------------ on the GPU
def _assert_sums_close(got, ref, n_z, n_nhi, rtol=1e-12):
    g, r = api.unpack_dla_statistics(got, n_z, n_nhi), api.unpack_dla_statistics(ref, n_z, n_nhi)
    for k in ("counts", "dla", "nhi"):
        assert np.all(np.abs(g[k] - r[k]) <= rtol * np.abs(r[k])), (k, np.max(np.abs(g[k] - r[k])))
    # q (1 - q) cancels where q is near 1; d/dq q (1 - q) is at most 1, so its error is that of q: the scale is sum q
    for k, mean in (("counts_var", "counts"), ("dla_var", "dla")):
        assert np.all(np.abs(g[k] - r[k]) <= rtol * (np.abs(r[k]) + r[mean])), (k, np.max(np.abs(g[k] - r[k])))
    # e2 - e^2 cancels where one sample carries the weight: compare on the scale of sum e2 >= nhi_var
    scale = r["nhi_var"] + r["nhi"] ** 2
    assert np.all(np.abs(g["nhi_var"] - r["nhi_var"]) <= rtol * scale), "nhi_var"
    assert np.all(np.abs(g["path"] - r["path"]) <= 1e-14 * np.abs(r["path"])), "path"
    assert g["num_quasars"] == r["num_quasars"]


def _random_edges(rng, lo, hi, n):
    return np.sort(rng.uniform(lo, hi, n + 1))


@pytest.fixture(scope="module")
def processed():
    """process_device outputs of 300 synthetic quasars with the 10 000 default samples."""
    import torch
    from gp_dla_detection_b200 import synthetic as syn
    model = syn.make_model()
    samples = syn.make_samples(10000)
    proc = api.DLAProcessor(model, samples, syn.make_prior(), device=0)
    pad = api.pad_spectra(syn.make_spectra(model, 300, seed=11, dla_fraction=0.3))
    up = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dtype=dt)).cuda()
    out = proc.process_device(up(pad["wavelengths"], np.float64), up(pad["flux"], np.float64),
                              up(pad["noise_variance"], np.float64), up(pad["pixel_mask"], np.uint8),
                              up(pad["lengths"], np.int32), up(pad["z_qsos"], np.float64),
                              return_sample_log_likelihoods=True)
    host = {k: v.cpu().numpy() for k, v in out.items()}
    yield dict(proc=proc, samples=samples, out=out, host=host)
    proc.close()


def _oracle(host, samples, z_edges, n_edges, select=None, **kw):
    return O.dla_statistics_sums(host["sample_log_likelihoods_dla"], host["p_dlas"], host["min_z_dlas"],
                                 host["max_z_dlas"], samples["offset_samples"], samples["log_nhi_samples"],
                                 samples["nhi_samples"], z_edges, n_edges, select=select, **kw)


@pytest.mark.gpu
def test_kernel_matches_oracle_on_processed_quasars(processed):
    import torch
    rng = np.random.default_rng(5)
    host, samples = processed["host"], processed["samples"]
    Q = host["p_dlas"].size
    zlo, zhi = np.nanmin(host["min_z_dlas"]), np.nanmax(host["max_z_dlas"])
    for trial, (n_z, n_nhi) in enumerate(((1, 1), (5, 30), (7, 13))):
        z_edges = _random_edges(rng, zlo - 0.1, zhi + 0.1, n_z)
        n_edges = _random_edges(rng, 19.8, 24.0, n_nhi)
        select = rng.random(Q) < 0.8 if trial else None
        ref = _oracle(host, samples, z_edges, n_edges, select=select)
        sel_t = None if select is None else torch.from_numpy(select).cuda()
        got = processed["proc"].statistics_device(processed["out"], z_edges, n_edges, select=sel_t).cpu().numpy()
        _assert_sums_close(got, ref, n_z, n_nhi)
        assert ref[-1] > 0.5 * Q


@pytest.mark.gpu
def test_bin_membership_on_exact_boundaries():
    """Edges on exactly computed z_ij and stored log N_j; one sample carries the weight of each quasar, so a membership
    difference would show as a whole-weight difference."""
    rng = np.random.default_rng(8)
    S, Q = 97, 24
    off = rng.random(S)
    lnhi = rng.uniform(20.0, 22.5, S)
    nhi = 10.0 ** lnhi
    zlo, zhi = np.full(Q, 2.3), np.full(Q, 3.1)
    z = zlo[0] + (zhi[0] - zlo[0]) * off                       # the kernel's rounding
    top = rng.choice(S, Q, replace=False)
    ll = np.full((Q, S), -40.0)
    ll[np.arange(Q), top] = 0.0
    p = rng.uniform(0.5, 1.0, Q)
    for k in range(4):
        zs = np.unique(np.concatenate([[2.0, 3.5], z[top[k * 6:k * 6 + 3]]]))
        ns = np.unique(np.concatenate([[19.0, 23.0], lnhi[top[k * 6 + 3:k * 6 + 6]]]))
        thr = float(lnhi[top[(k * 5 + 1) % Q]])
        ref = O.dla_statistics_sums(ll, p, zlo, zhi, off, lnhi, nhi, zs, ns, dla_log_nhi_min=thr)
        got = api.dla_statistics_sums(dict(sample_log_likelihoods_dla=ll, p_dlas=p, min_z_dlas=zlo, max_z_dlas=zhi),
                                      dict(offset_samples=off, log_nhi_samples=lnhi, nhi_samples=nhi), zs, ns,
                                      dla_log_nhi_min=thr)
        _assert_sums_close(got, ref, zs.size - 1, ns.size - 1)


@pytest.mark.gpu
def test_large_sample_count_through_l2():
    """S = 100 000 does not fit in shared memory: the kernel reads each row through the permutation."""
    from gp_dla_detection_b200 import synthetic as syn
    rng = np.random.default_rng(9)
    samples = syn.make_samples(100000)
    Q, S = 12, 100000
    ll = -0.5 * rng.standard_normal((Q, S)) ** 2 * 20 - 3.0 * rng.random((Q, 1))
    p = rng.random(Q)
    zlo = rng.uniform(2.0, 3.0, Q)
    zhi = zlo + rng.uniform(0.2, 1.5, Q)
    res = dict(sample_log_likelihoods_dla=ll, p_dlas=p, min_z_dlas=zlo, max_z_dlas=zhi)
    z_edges, n_edges = np.linspace(2.0, 4.5, 6), np.linspace(20.0, 23.0, 31)
    got = api.dla_statistics_sums(res, samples, z_edges, n_edges)
    ref = O.dla_statistics_sums(ll, p, zlo, zhi, samples["offset_samples"], samples["log_nhi_samples"],
                                samples["nhi_samples"], z_edges, n_edges)
    _assert_sums_close(got, ref, 5, 30)


@pytest.mark.gpu
def test_repeatable_host_equals_device_and_halves_add(processed):
    import torch
    host, samples, proc, out = processed["host"], processed["samples"], processed["proc"], processed["out"]
    z_edges, n_edges = np.linspace(1.9, 5.0, 6), np.linspace(20.0, 23.0, 31)
    a = proc.statistics_device(out, z_edges, n_edges).cpu().numpy()
    b = proc.statistics_device(out, z_edges, n_edges).cpu().numpy()
    assert a.tobytes() == b.tobytes()
    h = api.dla_statistics_sums(host, samples, z_edges, n_edges)
    assert h.tobytes() == a.tobytes()
    Q = host["p_dlas"].size
    half = {k: v[:Q // 2] for k, v in out.items()}
    rest = {k: v[Q // 2:].contiguous() for k, v in out.items()}
    acc = proc.statistics_device(half, z_edges, n_edges)
    acc = proc.statistics_device(rest, z_edges, n_edges, sums=acc).cpu().numpy()
    _assert_sums_close(acc, a, 5, 30, rtol=1e-13)


@pytest.mark.gpu
def test_end_to_end_expected_dla_count_matches_injected():
    import torch
    from gp_dla_detection_b200 import synthetic as syn
    model = syn.make_model()
    samples = syn.make_samples(10000)
    spectra = syn.make_spectra(model, 2000, seed=21, dla_fraction=0.3)
    pad = api.pad_spectra(spectra)
    proc = api.DLAProcessor(model, samples, syn.make_prior(), device=0)
    try:
        up = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dtype=dt)).cuda()
        out = proc.process_device(up(pad["wavelengths"], np.float64), up(pad["flux"], np.float64),
                                  up(pad["noise_variance"], np.float64), up(pad["pixel_mask"], np.uint8),
                                  up(pad["lengths"], np.int32), up(pad["z_qsos"], np.float64),
                                  return_sample_log_likelihoods=True)
        # one cell each: the variance of a cell is exact, that of a sum of one quasar's cells is not a sum of variances
        every = api.unpack_dla_statistics(proc.statistics_device(out, [0.0, 10.0], [20.0, 30.0]), 1, 1)
        high = api.unpack_dla_statistics(proc.statistics_device(out, [0.0, 10.0], [20.5, 30.0]), 1, 1)
    finally:
        proc.close()
    # every injected system and every sample has log N >= 20, so the first cell counts all of them; above 20.5 the
    # steep sample prior moves posterior weight below the cut, and that count is reported, not asserted
    total, sigma_total = every["counts"][0, 0], math.sqrt(every["counts_var"][0, 0])
    injected_total = int(np.count_nonzero(np.isfinite(spectra["truth_log_nhi"])))
    injected_high = int(np.count_nonzero(spectra["truth_log_nhi"] >= 20.5))
    print("end-to-end: expected %.2f +- %.2f DLAs (log N >= 20), injected %d; expected %.2f +- %.2f with log N >= 20.5, "
          "injected %d; %d quasars contribute" % (total, sigma_total, injected_total, high["counts"][0, 0],
                                                  math.sqrt(high["counts_var"][0, 0]), injected_high,
                                                  int(every["num_quasars"])))
    assert abs(total - injected_total) <= 4 * sigma_total + 0.05 * injected_total
