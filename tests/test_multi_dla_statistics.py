"""Population statistics of the multi-DLA catalogue (Ho et al. 2021): the NumPy restatement pinned by hand values, its
reduction to the single-DLA statistic and the mixture identities on the CPU, the C entries' argument checks, the sharded
sum, and on the GPU the device twin of process_multi and the statistics kernel against the restatement."""
import ctypes
import math
import os
import socket

import numpy as np
import pytest

from gp_dla_detection_b200 import _lib, api
from gp_dla_detection_b200 import sharding as sh
from oracle import dla_statistics_oracle as O1
from oracle import multi_dla_statistics_oracle as O


def _assert_sums_close(got, ref, n_z, n_nhi, rtol=1e-12):
    """Each part within rtol of its scale (as the single-DLA tests compare), path within 1e-14, num_quasars exact."""
    g, r = api.unpack_dla_statistics(got, n_z, n_nhi), api.unpack_dla_statistics(ref, n_z, n_nhi)
    for k in ("counts", "dla", "nhi"):
        assert np.all(np.abs(g[k] - r[k]) <= rtol * np.abs(r[k])), (k, np.max(np.abs(g[k] - r[k])))
    # E[X^2] - E[X]^2 cancels where one outcome carries the weight: compare on the scale of E[X^2] <= J E[X]
    for k, mean in (("counts_var", "counts"), ("dla_var", "dla")):
        scale = np.abs(r[k]) + 4 * r[mean] + r[mean] ** 2
        assert np.all(np.abs(g[k] - r[k]) <= rtol * scale), (k, np.max(np.abs(g[k] - r[k])))
    scale = np.abs(r["nhi_var"]) + r["nhi"] ** 2
    assert np.all(np.abs(g["nhi_var"] - r["nhi_var"]) <= rtol * scale), "nhi_var"
    assert np.all(np.abs(g["path"] - r["path"]) <= 1e-14 * np.abs(r["path"])), "path"
    assert g["num_quasars"] == r["num_quasars"]


# ------------------------------------------------------------------ the restatement, by hand
def _hand_quasar():
    """One quasar, J = 2, four samples on z in [2, 3] (z = 2 + offset)."""
    offset = np.array([0.1, 0.2, 0.7, 0.3])                     # z = 2.1, 2.2, 2.7, 2.3
    log_nhi = np.array([20.5, 20.6, 21.5, 20.4])
    ll = np.array([np.log([1.0, 2.0, 1.0, 4.0]),                 # level 1: w = 1/8, 2/8, 1/8, 4/8
                   [np.log(2.0), 0.0, 0.0, np.nan]])             # level 2: w = 2/4, 1/4, 1/4, 0 (filtered)
    part = np.array([[1, 2, 0, 0]])                              # level 2 places sample i and sample part[0, i]
    post = np.array([0.1, 0.2, 0.3, 0.4])                        # no DLA, sub-DLA, 1 DLA, 2 DLAs
    return ll, part, post, offset, log_nhi, 10.0 ** log_nhi


def test_oracle_known_answer_one_quasar():
    ll, part, post, off, lnhi, nhi = _hand_quasar()
    z_edges, n_edges = [2.0, 2.5, 3.0], [20.0, 21.0, 22.0]
    sums = O.multi_dla_statistics_sums(ll[None], part[None], post[None], [2.0], [3.0], off, lnhi, nhi, z_edges, n_edges)
    t = api.unpack_dla_statistics(sums, 2, 2)
    p1, p2 = 0.3, 0.4
    # cell (z bin 0, log-N bin 0) holds samples 0, 1, 3.  Level 1: one absorber, X in {0, 1}.  Level 2: sample 0
    # places both absorbers in it (X = 2), samples 1 and 2 one each (the other one of sample 1 is in z bin 1)
    e00 = p1 * 7 / 8 + p2 * (2 * 2 / 4 + 1 / 4 + 1 / 4)
    e200 = p1 * 7 / 8 + p2 * (4 * 2 / 4 + 1 / 4 + 1 / 4)
    e11 = p1 * 1 / 8 + p2 * (1 / 4 + 1 / 4)                      # sample 2 (z 2.7, log N 21.5)
    ref = np.zeros((2, 2))
    ref[0, 0], ref[1, 1] = e00, e11
    np.testing.assert_allclose(t["counts"], ref, rtol=1e-15, atol=0)
    np.testing.assert_allclose(t["counts_var"], [[e200 - e00 ** 2, 0], [0, e11 - e11 ** 2]], rtol=1e-14, atol=0)
    # every sample is a DLA (log N >= 20.3): D of z bin 0 is X of cell (0, 0)
    np.testing.assert_allclose(t["dla"], [e00, e11], rtol=1e-15)
    np.testing.assert_allclose(t["dla_var"], [e200 - e00 ** 2, e11 - e11 ** 2], rtol=1e-14)
    N0, N1, N2, N3 = nhi
    e = p1 * (N0 / 8 + 2 * N1 / 8 + 4 * N3 / 8) + p2 * ((N0 + N1) * 2 / 4 + N1 / 4 + N0 / 4)
    e2 = p1 * (N0 ** 2 / 8 + 2 * N1 ** 2 / 8 + 4 * N3 ** 2 / 8) + p2 * ((N0 + N1) ** 2 * 2 / 4 + N1 ** 2 / 4 + N0 ** 2 / 4)
    np.testing.assert_allclose(t["nhi"], [e, p1 * N2 / 8 + p2 * N2 / 2], rtol=1e-14)
    np.testing.assert_allclose(t["nhi_var"][0], e2 - e * e, rtol=1e-13)
    np.testing.assert_allclose(t["path"], [O1.path_length(2, 3, 2, 2.5, 0.3), O1.path_length(2, 3, 2.5, 3, 0.3)],
                               rtol=1e-15)
    assert t["num_quasars"] == 1.0


@pytest.mark.parametrize("why", ["select", "nan_posterior", "empty_z", "all_nan_level", "partner_out_of_range"])
def test_oracle_excluded_quasar_contributes_nothing(why):
    ll, part, post, off, lnhi, nhi = _hand_quasar()
    zhi, sel = 3.0, None
    if why == "select":
        sel = [False]
    elif why == "nan_posterior":
        post = post.copy(); post[0] = np.nan
    elif why == "empty_z":
        zhi = 2.0
    elif why == "all_nan_level":
        ll = ll.copy(); ll[1] = np.nan
    else:
        part = part.copy(); part[0, 2] = 4
    sums = O.multi_dla_statistics_sums(ll[None], part[None], post[None], [2.0], [zhi], off, lnhi, nhi,
                                       [2.0, 2.5, 3.0], [20.0, 21.0], select=sel)
    assert np.array_equal(sums, np.zeros(api.dla_statistics_width(2, 1)))


def test_oracle_skips_levels_without_weight():
    """A level with p_j == 0 is skipped: its NaN row and out-of-range partners do not exclude the quasar."""
    ll, part, post, off, lnhi, nhi = _hand_quasar()
    ll2, part2, post2 = ll.copy(), part.copy(), post.copy()
    ll2[1] = np.nan
    part2[0] = -7
    post2[3] = 0.0
    a = O.multi_dla_statistics_sums(ll2[None], part2[None], post2[None], [2.0], [3.0], off, lnhi, nhi, [2.0, 3.0],
                                    [20.0, 22.0])
    b = O.multi_dla_statistics_sums(ll[:1][None], None, post[:3][None], [2.0], [3.0], off, lnhi, nhi, [2.0, 3.0],
                                    [20.0, 22.0])
    assert np.array_equal(a, b) and a[-1] == 1.0


def _random_case(rng, Q, J, S, nan_fraction=0.1):
    ll = -0.5 * (rng.standard_normal((Q, J, S)) * 4) ** 2 - 3.0 * rng.random((Q, J, 1))
    ll[:, 1:][rng.random((Q, J - 1, S)) < nan_fraction] = np.nan
    part = rng.integers(0, S, (Q, J - 1, S)).astype(np.int32)
    post = rng.random((Q, J + 2)) ** 2
    post /= post.sum(axis=1, keepdims=True)
    zlo = rng.uniform(2.0, 3.0, Q)
    zhi = zlo + rng.uniform(0.2, 1.5, Q)
    lnhi = rng.uniform(20.0, 23.0, S)
    return ll, part, post, zlo, zhi, rng.random(S), lnhi, 10.0 ** lnhi


def test_one_level_is_the_single_dla_statistic():
    rng = np.random.default_rng(2)
    Q, S = 9, 80
    ll, _, _, zlo, zhi, off, lnhi, nhi = _random_case(rng, Q, 1, S)
    p = rng.random(Q)
    p[3] = 1.0 - 1e-12                                          # q (1 - q) and q - q^2 round differently near 1
    post = np.stack([1.0 - p, np.zeros(Q), p], axis=1)
    z_edges, n_edges = [2.0, 2.4, 3.1, 4.6], [20.0, 20.5, 21.7, 23.0]
    got = O.multi_dla_statistics_sums(ll, None, post, zlo, zhi, off, lnhi, nhi, z_edges, n_edges)
    ref = O1.dla_statistics_sums(ll[:, 0], p, zlo, zhi, off, lnhi, nhi, z_edges, n_edges)
    _assert_sums_close(got, ref, 3, 3, rtol=1e-14)


def test_consistency_identity_one_cell():
    """One z bin over every absorber and one log-N bin over every sample: X is the number of DLAs, whose law is the
    model posterior: E[X] = sum_j j p_j, Var[X] = sum_j j^2 p_j - (sum_j j p_j)^2."""
    rng = np.random.default_rng(4)
    Q, J, S = 7, 4, 60
    ll, part, post, zlo, zhi, off, lnhi, nhi = _random_case(rng, Q, J, S)
    sums = O.multi_dla_statistics_sums(ll, part, post, zlo, zhi, off, lnhi, nhi, [0.0, 10.0], [19.0, 30.0],
                                       dla_log_nhi_min=19.5)
    t = api.unpack_dla_statistics(sums, 1, 1)
    j = np.arange(1, J + 1)
    mean = post[:, 2:] @ j
    var = post[:, 2:] @ (j * j) - mean ** 2
    assert abs(t["counts"][0, 0] - mean.sum()) <= 1e-12 * mean.sum()
    assert abs(t["counts_var"][0, 0] - var.sum()) <= 1e-12 * mean.sum()
    assert t["dla"][0] == t["counts"][0, 0] and t["num_quasars"] == Q


# ------------------------------------------------------------------ the C entries' argument checks (no GPU needed)
def _call_host(max_dlas=2, part=None, null_part=False, z_edges=(2.0, 2.5, 3.0), device=False, Q=1, S=4):
    lib = _lib.load()
    J = max(max_dlas, 1)
    ll, post = np.zeros((Q, J, S)), np.full((Q, J + 2), 1.0 / (J + 2))
    zlo, zhi = np.full(Q, 2.0), np.full(Q, 3.0)
    if part is None:
        part = np.zeros((Q, max(J - 1, 1), S), dtype=np.int32)
    part = np.ascontiguousarray(part, dtype=np.int32)
    off, lnhi, nhi = np.linspace(0, 1, S), np.full(S, 21.0), np.full(S, 1e21)
    ze, ne = np.asarray(z_edges, float), np.array([20.0, 21.0, 22.0])
    sums = np.zeros(api.dla_statistics_width(ze.size - 1, ne.size - 1))
    vp = lambda a: ctypes.c_void_p(a.ctypes.data)
    args = [Q, S, max_dlas, vp(ll), None if null_part else vp(part), vp(post), vp(zlo), vp(zhi), None, vp(off),
            vp(lnhi), vp(nhi), ze.size - 1, api._dp(ze), ne.size - 1, api._dp(ne), 20.3, 0.3, vp(sums)]
    rc = lib.gpdla_multi_dla_statistics_device(*args, None) if device else lib.gpdla_multi_dla_statistics(*args)
    return rc, (lib.gpdla_last_error(None) or b"").decode()


@pytest.mark.parametrize("device", [False, True])
@pytest.mark.parametrize("case", ["max_dlas_zero", "max_dlas_five", "null_partners", "unsorted_z"])
def test_c_entries_reject_bad_arguments(case, device):
    kw = dict(device=device)
    if case == "max_dlas_zero":
        kw["max_dlas"] = 0
    elif case == "max_dlas_five":
        kw["max_dlas"] = 5
    elif case == "null_partners":
        kw["null_part"] = True
    else:
        kw["z_edges"] = (2.0, 3.0, 2.5)
    rc, msg = _call_host(**kw)
    assert rc == _lib.GPDLA_ERR_INVALID, (rc, msg)
    name = "gpdla_multi_dla_statistics_device" if device else "gpdla_multi_dla_statistics"
    assert msg.startswith(name + ": "), msg


@pytest.mark.parametrize("bad", [-1, 4])
def test_host_entry_rejects_partner_out_of_range(bad):
    part = np.zeros((1, 2, 4), dtype=np.int32)
    part[0, 1, 3] = bad
    rc, msg = _call_host(max_dlas=3, part=part)
    assert rc == _lib.GPDLA_ERR_INVALID, (rc, msg)
    assert msg.startswith("gpdla_multi_dla_statistics: base_sample_inds[0][1][3]"), msg


def test_one_level_needs_no_partners():
    """max_dlas == 1 with NULL base_sample_inds passes the checks (the call then needs a device)."""
    import torch
    rc, msg = _call_host(max_dlas=1, null_part=True)
    assert rc == (_lib.GPDLA_OK if torch.cuda.is_available() else _lib.GPDLA_ERR_CUDA), msg


# ------------------------------------------------------------------ sharded sum, 2 gloo ranks, CPU stand-in
Z_EDGES, N_EDGES = [2.0, 2.6, 3.4, 6.0], [20.0, 20.5, 21.0, 22.0, 23.0]
S_STAND_IN, J_STAND_IN = 48, 3


def _stand_in_samples(S=S_STAND_IN):
    lnhi = 20.0 + 3.0 * ((np.arange(S) * 0.618034) % 1.0)
    return (np.arange(S) + 0.5) / S, lnhi, 10.0 ** lnhi


def _stand_in_results(sp, S=S_STAND_IN, J=J_STAND_IN):
    """Deterministic per-quasar stand-ins for process_multi_device outputs, keyed on z_qso."""
    z = np.asarray(sp["z_qsos"])
    off = (np.arange(S) + 0.5) / S
    frac = np.modf(7.0 * z)[0]
    ll = -30.0 * (off[None, None, :] - frac[:, None, None] * np.arange(1, J + 1)[None, :, None] / J) ** 2
    part = ((np.arange(S)[None, None, :] * 7 + 5 * np.arange(1, J)[None, :, None] + (13 * z).astype(int)[:, None, None])
            % S).astype(np.int32)
    post = np.stack([1.0 + 0 * z, 0.5 + frac, 1 + z, 2.0 - frac, frac + 0.1], axis=1)
    post /= post.sum(axis=1, keepdims=True)
    return ll, part, post, z - 1.0, z - 0.05


def _stats_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from gp_dla_detection_b200 import synthetic as syn
    spectra = syn.make_spectra(syn.make_model(), 11, seed=6)
    select = np.arange(11) % 4 != 1
    off, lnhi, nhi = _stand_in_samples()

    def compute(sp, sel, sums):
        ll, part, post, zlo, zhi = _stand_in_results(sp)
        return O.multi_dla_statistics_sums(ll, part, post, zlo, zhi, off, lnhi, nhi, Z_EDGES, N_EDGES, select=sel,
                                           sums=sums)
    res = sh.multi_dla_statistics_sharded(None, None, spectra, None, Z_EDGES, N_EDGES, select=select,
                                          max_dlas=J_STAND_IN, batch_quasars=2, compute=compute)
    q.put((rank, res["sums"].tobytes(), res["blocks"]))
    dist.destroy_process_group()


def test_sharded_multi_statistics_two_gloo_ranks():
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
    assert (r0, r1) == (0, 1) and b0 == b1
    total = np.frombuffer(b0, dtype=np.float64)
    spectra = syn.make_spectra(syn.make_model(), 11, seed=6)
    select = np.arange(11) % 4 != 1
    off, lnhi, nhi = _stand_in_samples()
    ranks = []
    for s0, e0 in blocks:
        acc = np.zeros(api.dla_statistics_width(3, 4))
        for a in range(s0, e0, 2):
            ll, part, post, zlo, zhi = _stand_in_results(sh.slice_spectra(spectra, a, min(e0, a + 2)))
            acc = O.multi_dla_statistics_sums(ll, part, post, zlo, zhi, off, lnhi, nhi, Z_EDGES, N_EDGES,
                                              select=select[a:a + 2], sums=acc)
        ranks.append(acc)
    assert np.array_equal(total, ranks[0] + ranks[1])
    # the one-process oracle over the whole catalogue: the same sums up to the order of the additions
    ll, part, post, zlo, zhi = _stand_in_results(spectra)
    whole = O.multi_dla_statistics_sums(ll, part, post, zlo, zhi, off, lnhi, nhi, Z_EDGES, N_EDGES, select=select)
    _assert_sums_close(total, whole, 3, 4, rtol=1e-13)
    assert total[-1] == np.count_nonzero(select)


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
    """process_multi_device outputs (J = 4) of 240 synthetic mean-flux spectra, some with two injected DLAs, with the
    10 000 default samples."""
    from gp_dla_detection_b200 import synthetic as syn
    model = syn.make_model()
    samples = syn.make_samples(10000, with_lls=True)
    spectra = syn.make_spectra(model, 240, seed=12, dla_fraction=0.4, meanflux=True, second_dla_fraction=0.4)
    proc = api.DLAProcessor(model, samples, syn.make_prior(), device=0)
    out = proc.process_multi_device(*_planes(spectra), max_dlas=4, return_samples=True)
    host = {k: v.cpu().numpy() for k, v in out.items()}
    yield dict(proc=proc, samples=samples, spectra=spectra, out=out, host=host, model=model)
    proc.close()


def _oracle(host, samples, z_edges, n_edges, select=None, **kw):
    return O.multi_dla_statistics_sums(host["sample_log_likelihoods_dla"], host["base_sample_inds"],
                                       host["model_posteriors"], host["min_z_dlas"], host["max_z_dlas"],
                                       samples["offset_samples"], samples["log_nhi_samples"], samples["nhi_samples"],
                                       z_edges, n_edges, select=select, **kw)


@pytest.mark.gpu
def test_process_multi_device_matches_process_multi(processed):
    from gp_dla_detection_b200 import synthetic as syn
    sp = {k: (v[:60] if isinstance(v, (list, np.ndarray)) else v) for k, v in processed["spectra"].items()}
    ref = processed["proc"].process_multi(sp, max_dlas=4, return_samples=True)
    host = processed["host"]
    for k, v in ref.items():
        got = host[k][:60]
        if k in ("sample_log_likelihoods_dla", "base_sample_inds"):
            got = np.transpose(got, (0, 2, 1))
        assert got.shape == v.shape and got.dtype == v.dtype, k
        assert np.array_equal(got, v, equal_nan=True), k
    assert np.count_nonzero(np.argmax(host["model_posteriors"], axis=1) >= 3) > 0   # two-DLA quasars are found


@pytest.mark.gpu
def test_kernel_matches_oracle_on_processed_quasars(processed):
    import torch
    rng = np.random.default_rng(5)
    host, samples = processed["host"], processed["samples"]
    Q = host["min_z_dlas"].size
    zlo, zhi = np.nanmin(host["min_z_dlas"]), np.nanmax(host["max_z_dlas"])
    for n_z, n_nhi in ((1, 1), (5, 30), (7, 13)):
        z_edges = np.sort(rng.uniform(zlo - 0.1, zhi + 0.1, n_z + 1))
        n_edges = np.sort(rng.uniform(19.8, 24.0, n_nhi + 1))
        for select in (None, rng.random(Q) < 0.8):
            ref = _oracle(host, samples, z_edges, n_edges, select=select)
            sel_t = None if select is None else torch.from_numpy(select).cuda()
            got = processed["proc"].multi_statistics_device(processed["out"], z_edges, n_edges,
                                                            select=sel_t).cpu().numpy()
            _assert_sums_close(got, ref, n_z, n_nhi)
            assert ref[-1] > 0.5 * Q


@pytest.mark.gpu
def test_bin_membership_on_exact_partner_boundaries():
    """Edges on exactly computed z and stored log N of the partner absorbers of a dominating level-2 / level-3 sample;
    one sample carries each level's weight, so a membership difference shows as a whole-weight difference."""
    rng = np.random.default_rng(8)
    S, Q, J = 97, 24, 3
    off = rng.random(S)
    lnhi = rng.uniform(20.0, 22.5, S)
    nhi = 10.0 ** lnhi
    zlo, zhi = np.full(Q, 2.3), np.full(Q, 3.1)
    z = zlo[0] + (zhi[0] - zlo[0]) * off                        # the kernel's rounding
    top = rng.choice(S, Q, replace=False)
    ll = np.full((Q, J, S), -40.0)
    ll[np.arange(Q), :, top] = 0.0
    part = rng.integers(0, S, (Q, J - 1, S)).astype(np.int32)
    post = np.zeros((Q, J + 2))
    post[:, 0] = 0.05
    post[:, 3] = rng.uniform(0.2, 0.5, Q)
    post[:, 4] = 0.95 - post[:, 3]
    partners = part[np.arange(Q), :, top]                       # [Q, J - 1]: where the dominating samples' partners sit
    samples = dict(offset_samples=off, log_nhi_samples=lnhi, nhi_samples=nhi)
    res = dict(sample_log_likelihoods_dla=np.transpose(ll, (0, 2, 1)), base_sample_inds=np.transpose(part, (0, 2, 1)),
               model_posteriors=post, min_z_dlas=zlo, max_z_dlas=zhi)
    for k in range(4):
        sl = slice(k * 6, k * 6 + 6)
        zs = np.unique(np.concatenate([[2.0, 3.5], z[partners[sl, 0]], z[partners[sl.start:sl.start + 2, 1]]]))
        ns = np.unique(np.concatenate([[19.0, 23.0], lnhi[partners[sl, 1]], lnhi[partners[sl.start + 3:sl.stop, 0]]]))
        thr = float(lnhi[partners[(k * 5 + 1) % Q, 0]])
        ref = O.multi_dla_statistics_sums(ll, part, post, zlo, zhi, off, lnhi, nhi, zs, ns, dla_log_nhi_min=thr)
        got = api.multi_dla_statistics_sums(res, samples, zs, ns, dla_log_nhi_min=thr)
        _assert_sums_close(got, ref, zs.size - 1, ns.size - 1)


@pytest.mark.gpu
def test_one_level_matches_single_dla_entry(processed):
    import torch
    proc, out, host = processed["proc"], processed["out"], processed["host"]
    ll0 = host["sample_log_likelihoods_dla"][:, 0]
    p = host["model_posteriors"][:, 2].copy()
    keep = np.flatnonzero(np.all(np.isfinite(ll0), axis=1) & np.isfinite(p))
    assert keep.size > 100
    idx = torch.from_numpy(keep).cuda()
    pt = torch.from_numpy(p).cuda()[idx]
    one = dict(sample_log_likelihoods_dla=out["sample_log_likelihoods_dla"][idx, :1].contiguous(),
               model_posteriors=torch.stack([1.0 - pt, torch.zeros_like(pt), pt], dim=1).contiguous(),
               min_z_dlas=out["min_z_dlas"][idx].contiguous(), max_z_dlas=out["max_z_dlas"][idx].contiguous())
    single = dict(sample_log_likelihoods_dla=out["sample_log_likelihoods_dla"][idx, 0].contiguous(), p_dlas=pt,
                  min_z_dlas=one["min_z_dlas"], max_z_dlas=one["max_z_dlas"])
    z_edges, n_edges = np.linspace(1.9, 5.0, 6), np.linspace(20.0, 23.0, 31)
    got = proc.multi_statistics_device(one, z_edges, n_edges).cpu().numpy()
    ref = proc.statistics_device(single, z_edges, n_edges).cpu().numpy()
    _assert_sums_close(got, ref, 5, 30, rtol=1e-13)


@pytest.mark.gpu
def test_consistency_identity_on_processed_quasars(processed):
    host = processed["host"]
    t = api.unpack_dla_statistics(processed["proc"].multi_statistics_device(processed["out"], [0.0, 10.0],
                                                                            [19.0, 30.0]), 1, 1)
    post = host["model_posteriors"]
    ok = np.all(np.isfinite(post), axis=1) & (host["max_z_dlas"] > host["min_z_dlas"])
    j = np.arange(1, post.shape[1] - 1)
    mean = post[ok, 2:] @ j
    var = post[ok, 2:] @ (j * j) - mean ** 2
    assert t["num_quasars"] == np.count_nonzero(ok)
    assert abs(t["counts"][0, 0] - mean.sum()) <= 1e-12 * mean.sum()
    assert abs(t["counts_var"][0, 0] - var.sum()) <= 1e-12 * (mean.sum() + var.sum())


@pytest.mark.gpu
def test_large_sample_count():
    """S = 100 000: four rows of 800 KB per quasar, random partners."""
    from gp_dla_detection_b200 import synthetic as syn
    rng = np.random.default_rng(9)
    samples = syn.make_samples(100000)
    Q, J, S = 8, 4, 100000
    ll, part, post, zlo, zhi, _, _, _ = _random_case(rng, Q, J, S)
    res = dict(sample_log_likelihoods_dla=np.transpose(ll, (0, 2, 1)), base_sample_inds=np.transpose(part, (0, 2, 1)),
               model_posteriors=post, min_z_dlas=zlo, max_z_dlas=zhi)
    z_edges, n_edges = np.linspace(2.0, 4.5, 6), np.linspace(20.0, 23.0, 31)
    got = api.multi_dla_statistics_sums(res, samples, z_edges, n_edges)
    ref = O.multi_dla_statistics_sums(ll, part, post, zlo, zhi, samples["offset_samples"], samples["log_nhi_samples"],
                                      samples["nhi_samples"], z_edges, n_edges)
    _assert_sums_close(got, ref, 5, 30)


@pytest.mark.gpu
def test_repeatable_host_equals_device_and_halves_add(processed):
    host, samples, proc, out = processed["host"], processed["samples"], processed["proc"], processed["out"]
    z_edges, n_edges = np.linspace(1.9, 5.0, 6), np.linspace(20.0, 23.0, 31)
    a = proc.multi_statistics_device(out, z_edges, n_edges).cpu().numpy()
    b = proc.multi_statistics_device(out, z_edges, n_edges).cpu().numpy()
    assert a.tobytes() == b.tobytes()
    ref_layout = dict(host)
    ref_layout["sample_log_likelihoods_dla"] = np.transpose(host["sample_log_likelihoods_dla"], (0, 2, 1))
    ref_layout["base_sample_inds"] = np.transpose(host["base_sample_inds"], (0, 2, 1))
    h = api.multi_dla_statistics_sums(ref_layout, samples, z_edges, n_edges)
    assert h.tobytes() == a.tobytes()
    Q = host["min_z_dlas"].size
    half = {k: v[:Q // 2] for k, v in out.items()}
    rest = {k: v[Q // 2:].contiguous() for k, v in out.items()}
    acc = proc.multi_statistics_device(half, z_edges, n_edges)
    acc = proc.multi_statistics_device(rest, z_edges, n_edges, sums=acc).cpu().numpy()
    _assert_sums_close(acc, a, 5, 30, rtol=1e-13)


@pytest.mark.gpu
def test_end_to_end_expected_absorber_count_matches_injected():
    from gp_dla_detection_b200 import synthetic as syn
    model = syn.make_model()
    samples = syn.make_samples(10000, with_lls=True)
    spectra = syn.make_spectra(model, 2000, seed=21, dla_fraction=0.3, meanflux=True, second_dla_fraction=0.3)
    proc = api.DLAProcessor(model, samples, syn.make_prior(), device=0)
    try:
        out = proc.process_multi_device(*_planes(spectra), max_dlas=4, return_samples=True)
        # one cell: every injected system and every sample has log N >= 20
        every = api.unpack_dla_statistics(proc.multi_statistics_device(out, [0.0, 10.0], [20.0, 30.0]), 1, 1)
        post = out["model_posteriors"].cpu().numpy()
    finally:
        proc.close()
    total, sigma = every["counts"][0, 0], math.sqrt(every["counts_var"][0, 0])
    one = int(np.count_nonzero(np.isfinite(spectra["truth_log_nhi"])))
    two = int(np.count_nonzero(np.isfinite(spectra["truth_log_nhi2"])))
    injected = one + two
    ok = np.all(np.isfinite(post), axis=1)
    levels = post[ok, 2:].sum(axis=0)
    print("end-to-end: expected %.2f +- %.2f absorbers (log N >= 20), injected %d (%d spectra with one or more, %d "
          "with two); expected quasars per level 1..4: %s; sub-DLA %.2f; %d quasars contribute"
          % (total, sigma, injected, one, two, np.array2string(levels, precision=2), post[ok, 1].sum(),
             int(every["num_quasars"])))
    assert abs(total - injected) <= 4 * sigma + 0.05 * injected
