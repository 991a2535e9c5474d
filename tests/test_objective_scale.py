"""GP training objective (objective.m + spectrum_loss.m and the Lyman-series variant) at training-set scale.

objective_kernel is persistent: its grid holds at most SMs x resident CTAs, and each CTA walks the spectra
s = blockIdx.x, blockIdx.x + gridDim.x, ..., reusing its shared arrays and adding every spectrum into its own partial
gradient.  Every batch here has N = 16 SMs + 37 spectra, more than any resident grid (8 CTAs of 256 threads per SM at
most), so every CTA handles at least two spectra whatever the occupancy, and every edge row sits at an index of at
least 8 SMs, behind at least one ordinary spectrum of its CTA.  The reference is oracle/objective_oracle.py, compared
block by block: each column of dM and the dlog_omega block against that block's own largest entry."""
import contextlib
import ctypes

import numpy as np
import pytest

from oracle import objective_oracle as OB

try:
    from threadpoolctl import threadpool_limits
except ImportError:                        # the oracle is only slower without it
    threadpool_limits = None

CASES = {"k20": (20, 1217, 20), "k10": (10, 333, 10), "k40": (40, 200, 40)}   # k, num_pixels, seed
VARIANTS = ("plain", "lyseries")
POINTS = ("start", "iterate", "log_omega+3", "log_omega-8", "Mx30", "tau0=0.3,beta=5", "c0=1e-4", "c0=5")
F_BOUND, BLOCK_BOUND, SCALAR_BOUND = 1e-11, 1e-10, 1e-9
# Looser dM bounds at two extreme points.  The reference forms K^-1 M as D^-1 M - D^-1 M (C M) (spectrum_loss.m:55), the
# kernel as D^-1 M B^-1, the same matrix by Woodbury.  When M'D^-1 M >> I the reference's subtraction cancels digits:
# at log_omega - 8 the noise-variance-1e-6 row has d ~ 1e-6 (without that row the two orders agree to 2e-13), and
# M x 30 makes B ~ 900 times larger (cond B up to 3e4 for rows with about k pixels).  Measured on a B200 (1000 W),
# worst dM column against its own largest entry, worse of the two variants: log_omega - 8: k20 2.4e-8, k10 9.1e-9,
# k40 6.6e-7; M x 30: k20 3.3e-9, k10 8.3e-10, k40 7.3e-10.  The reference restated in the kernel's order (NumPy,
# B^-1 by LU) differs from it by 6.5e-9 (k20) and 5.0e-8 (k40) at log_omega - 8 and by 1.5e-9 and 1.6e-9 at M x 30.
# f, dlog_omega and the scalars keep their bounds there.
M_BOUNDS = {("log_omega-8", "k20"): 2e-7, ("log_omega-8", "k10"): 5e-8, ("log_omega-8", "k40"): 3e-6,
            ("Mx30", "k20"): 2e-8, ("Mx30", "k10"): 1e-8, ("Mx30", "k40"): 2e-8}


def one_blas_thread():
    """The oracle multiplies one spectrum's small matrices at a time, where a threaded BLAS is about ten times slower."""
    return threadpool_limits(1) if threadpool_limits else contextlib.nullcontext()


def forest_constants():
    """all_transition_wavelengths (Angstrom) and all_oscillator_strengths of multi_dlas/set_parameters_multi.m:76-142."""
    from oracle import process_qsos_oracle as O
    return O.TRANSITION_WAVELENGTHS * 1e8, O.OSCILLATOR_STRENGTHS


def lyseries_args(variant):
    return (31,) + forest_constants() if variant == "lyseries" else None


def edge_specs(P, k):
    """(name, observed columns, noise variance or None, flux outliers, keep 1 + z_qso in the last lya_1pzs column)."""
    rng = np.random.default_rng(P * 1000 + k)
    every = np.arange(P)
    specs = [("0 observed", every[:0], None, False, True)]
    for c in sorted({1, 2, k - 1, k, k + 1, 31, 32, 33, 64, 255, 256, 257}):        # around OBJ_TILE, OBJ_THREADS, k
        if c < P:
            specs.append(("%d observed" % c, np.sort(rng.choice(P, c, replace=False)), None, False, True))
    part = np.sort(rng.choice(P, (7 * P) // 10, replace=False))
    specs += [("column 0 only", every[:1], None, False, True),
              ("column P-1 only", every[-1:], None, False, True),
              ("fully observed", every, None, False, True),
              ("noise variance 1e-6", part, 1e-6, False, True),
              ("noise variance 1e4", part, 1e4, False, True),
              ("flux outliers +-50", every, None, True, True),
              # 1 + z_qso comes from the last lya_1pzs column (objective_lyseries.m:46), observed or not
              ("last column unobserved, z_qso kept", every[:-1], None, False, True),
              ("last column unobserved, z_qso NaN", every[:-1], None, False, False)]
    return specs


def scale_batch(sms, k, P, seed):
    """make_training_set with N = 16 SMs + 37 rows, most carrying 1 + z_qso in their last lya_1pzs column (a third keep
    NaN where it was not observed), the edge rows of edge_specs three apart from index 8 SMs + 5 on, and a last row
    without any observed pixel.  On the production grid the last column is at Lyman alpha and 1 + z_qso is its own
    1 + z; the shorter grids end in the forest, so their last column is set to 1 + z_qso, which keeps the higher
    series members below the quasar and in the model."""
    N = 16 * sms + 37
    x, y, lya, nv = OB.make_training_set(N, num_pixels=P, k=k, seed=seed)
    rest = 911.75 + 0.25 * np.arange(P)
    keep_nan = np.isnan(lya[:, -1]); keep_nan[::3] = False
    lya[:, -1] = np.where(keep_nan, lya[:, -1], np.nanmax(lya * 1215.6701 / rest, axis=1))
    rng = np.random.default_rng(seed + 7)
    M = x[:P * k].reshape(k, P).T
    om2 = np.exp(2 * x[P * k:P * (k + 1)])
    specs = edge_specs(P, k)
    rows = 8 * sms + 5 + 3 * np.arange(len(specs))
    assert rows[-1] < N - 1
    for r, (_, obs, var, outliers, zqso) in zip(rows, specs):
        z1 = (3.15 + rng.gamma(2.0, 0.3)) * rest / 1215.6701
        v = (0.1 + 0.4 * rng.random(P)) ** 2 if var is None else np.full(P, var)
        flux = M @ rng.standard_normal(k) + np.sqrt(v + om2 * 0.04) * rng.standard_normal(P)
        if outliers:
            out = rng.choice(P, 6, replace=False)
            flux[out] = np.where(np.arange(6) % 2 == 0, 50.0, -50.0)
        seen = np.zeros(P, bool); seen[obs] = True
        y[r] = np.where(seen, flux, np.nan); nv[r] = np.where(seen, v, np.nan); lya[r] = np.where(seen, z1, np.nan)
        lya[r, -1] = z1[-1] * 1215.6701 / rest[-1] if zqso else np.nan
    y[N - 1] = nv[N - 1] = lya[N - 1] = np.nan
    x[-3:] += [0.2, 0.1, -0.05]                # off the prior means, so every gradient block is exercised
    return dict(x=x, y=y, lya=lya, nv=nv, N=N, P=P, k=k, rows=rows, specs=specs)


def extreme_point(x, P, k, name):
    x = x.copy()
    om = slice(P * k, P * (k + 1))
    if name == "log_omega+3":
        x[om] += 3.0                           # omega^2 (absorption noise) dominates the pixel noise
    elif name == "log_omega-8":
        x[om] -= 8.0                           # the instrumental noise dominates
    elif name == "Mx30":
        x[:P * k] *= 30.0                      # B = I + M'D^-1 M large and less well conditioned
    elif name == "tau0=0.3,beta=5":
        x[-2:] = np.log([0.3, 5.0])            # exp(-tau) underflows to 0 at high z
    elif name == "c0=1e-4":
        x[-3] = np.log(1e-4)
    elif name == "c0=5":
        x[-3] = np.log(5.0)
    else:
        raise KeyError(name)
    return x


def prior_gradient(x):
    """The Kim et al. prior terms every evaluation adds to dlog_tau_0 and dlog_beta (objective.m:59-71)."""
    g = np.zeros_like(x)
    t0, beta = np.exp(x[-2:])
    g[-2] = t0 * (t0 - 0.0023) / 0.0007 ** 2
    g[-1] = beta * (beta - 3.65) / 0.21 ** 2
    return g


def block_errors(f, g, fr, gr, P, k):
    """f relative; every column of dM and the dlog_omega block against that block's own largest |entry|; the three
    scalars relative."""
    gm, rm = g[:P * k].reshape(k, P), gr[:P * k].reshape(k, P)
    om = slice(P * k, P * (k + 1))
    e = {"f": abs(f - fr) / abs(fr),
         "M": float(np.max(np.abs(gm - rm).max(axis=1) / np.abs(rm).max(axis=1))),
         "log_omega": float(np.abs(g[om] - gr[om]).max() / np.abs(gr[om]).max())}
    for name, i in (("c_0", -3), ("tau_0", -2), ("beta", -1)):
        e[name] = abs(g[i] - gr[i]) / abs(gr[i])
    return e


def assert_blocks(e, bounds=None, what=""):
    b = dict(f=F_BOUND, M=BLOCK_BOUND, log_omega=BLOCK_BOUND, c_0=SCALAR_BOUND, tau_0=SCALAR_BOUND, beta=SCALAR_BOUND)
    b.update(bounds or {})
    bad = {key: (e[key], b[key]) for key in b if not e[key] < b[key]}
    assert not bad, "%s: error above bound %s (all errors %s)" % (what, bad, e)


def blocks_close(f1, g1, f2, g2, P, k, tol):
    """Agreement of two GPU evaluations of one objective to tol, per block as in block_errors."""
    e = block_errors(f1, g1, f2, g2, P, k)
    bad = {key: v for key, v in e.items() if not v < tol}
    assert not bad, bad


# ---------------------------------------------------------------- CPU: the batch and the oracle on its edge rows
@pytest.mark.parametrize("sms", [148, 132, 114, 16])
def test_batch_places_every_edge_row_behind_an_ordinary_spectrum(sms):
    k, P, seed = CASES["k20"]
    b = scale_batch(sms, k, 333, seed)
    N, rows = b["N"], b["rows"]
    assert N == 16 * sms + 37 and N > 2 * 8 * sms                     # > 2 x any resident grid of 256-thread CTAs
    assert rows.min() >= 8 * sms                                      # row s runs on CTA s mod grid, grid <= 8 SMs
    observed = (~np.isnan(b["y"])).sum(axis=1)
    for r, (name, obs, *_) in zip(rows, b["specs"]):
        assert observed[r] == len(obs), name
    assert observed[N - 1] == 0
    ordinary = np.setdiff1d(np.arange(N), np.append(rows, N - 1))
    assert observed[ordinary].min() > 100
    counts = {len(s[1]) for s in b["specs"]}
    assert {0, 1, 2, 19, 20, 21, 31, 32, 33, 64, 255, 256, 257, 333} <= counts
    last = b["lya"][rows, -1]
    assert np.isnan(last).any() and np.isfinite(last).any()


@pytest.mark.parametrize("variant", VARIANTS)
def test_oracle_on_edge_rows_matches_dense_density(variant):
    """The reference on every edge row (1 pixel, fewer pixels than k, tiles, noise extremes, outliers, z_qso NaN)
    against the dense multivariate normal, and its gradient as the sum of the rows' gradients plus the prior."""
    from scipy.stats import multivariate_normal
    k, P = 4, 300
    b = scale_batch(4, k, P, 5)
    sel = np.append(b["rows"], b["N"] - 1)
    x, y, lya, nv = b["x"], b["y"][sel], b["lya"][sel], b["nv"][sel]
    ly = lyseries_args(variant)
    M = x[:P * k].reshape(k, P).T
    om2 = np.exp(2 * x[P * k:P * (k + 1)]); c0, t0, beta = np.exp(x[-3:])
    f, g = OB.objective(x, y, lya, nv, lyseries=ly)
    ref, gsum = 0.0, np.zeros_like(g)
    for i in range(len(sel)):
        ind = ~np.isnan(y[i])
        gsum += OB.objective(x, y[i:i + 1], lya[i:i + 1], nv[i:i + 1], priors=False, lyseries=ly)[1]
        if not ind.any():
            continue
        z1 = lya[i, ind]
        od = t0 * z1 ** beta
        if ly:
            nl, tw, osc = ly
            for l in range(1, nl):
                zl = tw[0] * z1 / tw[l]
                od = od + np.where(zl <= lya[i, -1], t0 * tw[l] * osc[l] / (tw[0] * osc[0]) * zl ** beta, 0.0)
        d = nv[i, ind] + om2[ind] * (1 - np.exp(-od) + c0) ** 2
        ref -= multivariate_normal.logpdf(y[i, ind], np.zeros(ind.sum()), M[ind] @ M[ind].T + np.diag(d))
    assert np.isfinite(f) and abs(f - ref) < 1e-9 * abs(ref)
    if ly:                                     # the series members below the quasar do enter on this short grid
        f0 = OB.objective(x, y, lya, nv)[0]
        assert abs(f - f0) > 1e-6 * abs(f0)
    gsum += prior_gradient(x)
    assert np.allclose(g, gsum, rtol=1e-12, atol=1e-12 * np.abs(g).max())


# ---------------------------------------------------------------- GPU fixtures (module scope: the oracle is a Python loop)
@pytest.fixture(scope="module")
def sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.fixture(scope="module")
def batch(sms):
    cache = {}

    def get(case):
        if case not in cache:
            cache[case] = scale_batch(sms, *CASES[case])
        return cache[case]
    return get


@pytest.fixture(scope="module")
def point(batch):
    """(case, variant, point name) -> x; the iterate is 15 L-BFGS iterations of learn_qso_model on that batch."""
    from gp_dla_detection_b200 import api
    cache = {}

    def get(case, variant, name):
        b = batch(case)
        if name == "start":
            return b["x"]
        if name != "iterate":
            return extreme_point(b["x"], b["P"], b["k"], name)
        if (case, variant) not in cache:
            ly = lyseries_args(variant) or (0, None, None)
            cache[case, variant] = api.learn_qso_model(b["y"], b["lya"], b["nv"], b["x"], b["k"], max_iter=15,
                                                       num_forest_lines=ly[0], all_transition_wavelengths=ly[1],
                                                       all_oscillator_strengths=ly[2])
        xi, _, res = cache[case, variant]
        assert res.nit >= 1 and not np.array_equal(xi, b["x"])
        return xi
    return get


def gpu_objective(b, x, variant):
    from gp_dla_detection_b200 import api
    ly = lyseries_args(variant) or (0, None, None)
    return api.objective_lyseries(x, b["y"], b["lya"], b["nv"], *ly)


def oracle_objective(b, x, variant, y=None, lya=None, nv=None):
    with one_blas_thread():
        return OB.objective(x, b["y"] if y is None else y, b["lya"] if lya is None else lya,
                            b["nv"] if nv is None else nv, lyseries=lyseries_args(variant))


# ---------------------------------------------------------------- GPU: the oracle at scale, every parameter point
@pytest.mark.gpu
@pytest.mark.parametrize("name", POINTS)
@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("case", list(CASES))
def test_scale_matches_oracle(batch, point, case, variant, name):
    b = batch(case)
    x = point(case, variant, name)
    f, g = gpu_objective(b, x, variant)
    fr, gr = oracle_objective(b, x, variant)
    e = block_errors(f, g, fr, gr, b["P"], b["k"])
    print("objective-scale %s %s %s N=%d: %s" % (case, variant, name, b["N"],
                                                  " ".join("%s=%.2e" % kv for kv in e.items())))
    looser = {"M": M_BOUNDS[name, case]} if (name, case) in M_BOUNDS else None
    assert_blocks(e, looser, what="%s %s %s" % (case, variant, name))


# ---------------------------------------------------------------- GPU: oracle-free properties at scale
@pytest.mark.gpu
@pytest.mark.parametrize("variant", VARIANTS)
def test_additivity_over_a_split_of_the_rows(batch, variant):
    """f(A u B) = f(A) + f(B); g(A u B) = g(A) + g(B) - prior, since every evaluation adds the Kim prior terms."""
    from gp_dla_detection_b200 import api
    b = batch("k20")
    x, P, k = b["x"], b["P"], b["k"]
    ly = lyseries_args(variant) or (0, None, None)
    ev = lambda rows: api.objective_lyseries(x, b["y"][rows], b["lya"][rows], b["nv"][rows], *ly)
    cut = 9 * (b["N"] // 16) + 11                                      # both halves hold edge rows
    f, g = ev(slice(None))
    fa, ga = ev(slice(0, cut))
    fb, gb = ev(slice(cut, None))
    f0, g0 = ev(slice(0, 0))                                           # no spectrum: the prior alone
    assert f0 == 0.0 and np.count_nonzero(g0[:-2]) == 0
    blocks_close(fa + fb, ga + gb - g0, f, g, P, k, 1e-12)


@pytest.mark.gpu
@pytest.mark.parametrize("variant", VARIANTS)
def test_row_permutation(batch, variant):
    """Permuting the rows moves spectra between CTAs and changes the order of the sums, not the result."""
    b = batch("k20")
    perm = np.random.default_rng(3).permutation(b["N"])
    f, g = gpu_objective(b, b["x"], variant)
    pb = dict(b, y=b["y"][perm], lya=b["lya"][perm], nv=b["nv"][perm])
    fp, gp = gpu_objective(pb, b["x"], variant)
    blocks_close(fp, gp, f, g, b["P"], b["k"], 1e-12)


@pytest.mark.gpu
@pytest.mark.parametrize("variant", VARIANTS)
def test_bit_reproducible_across_entries_and_streams(batch, variant):
    import torch
    from gp_dla_detection_b200 import api
    b = batch("k20")
    x = b["x"]
    f, g = gpu_objective(b, x, variant)
    f2, g2 = gpu_objective(b, x, variant)
    assert f2 == f and np.array_equal(g2, g)
    ly = lyseries_args(variant) or (0, None, None)
    dev = torch.device("cuda", 0)
    mats = [torch.from_numpy(b[key]).to(dev) for key in ("y", "lya", "nv")]
    ev = api.TrainingObjective(*mats, b["k"], num_forest_lines=ly[0], all_transition_wavelengths=ly[1],
                               all_oscillator_strengths=ly[2])
    try:
        for _ in range(2):
            fe, ge = ev(x)
            assert fe == f and np.array_equal(ge, g)
        side = torch.cuda.Stream(device=dev)
        xd = torch.from_numpy(x).to(dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            fd, gd = ev.evaluate_device(xd, stream=side.cuda_stream)
            fs, gs = fd.cpu().item(), gd.cpu().numpy()
        side.synchronize()
        assert fs == f and np.array_equal(gs, g)
    finally:
        ev.close()


@pytest.mark.gpu
@pytest.mark.parametrize("variant", VARIANTS)
def test_gpu_f_finite_differences(batch, variant):
    """Central differences of the GPU's own f along random directions, each supported on one block.  The tolerance is
    the rounding noise of the difference quotient, eps |f| / h (times a margin), plus the truncation error estimated
    from the quotient at 2h.  Lyman-series beta is left out: the reference's beta gradient uses log(1 + z_Lya) for
    every series member (spectrum_loss_lyseries.m:89) and is not the derivative of f."""
    from gp_dla_detection_b200 import api
    b = batch("k20")
    x, P, k = b["x"], b["P"], b["k"]
    ly = lyseries_args(variant) or (0, None, None)
    ev = api.TrainingObjective(b["y"], b["lya"], b["nv"], k, num_forest_lines=ly[0], all_transition_wavelengths=ly[1],
                               all_oscillator_strengths=ly[2])
    rng = np.random.default_rng(11)
    blocks = {"M": slice(0, P * k), "log_omega": slice(P * k, P * (k + 1)), "c_0": slice(-3, -2),
              "tau_0": slice(-2, -1)}
    if variant == "plain":
        blocks["beta"] = slice(-1, None)
    try:
        f, g = ev(x)
        g = g - prior_gradient(x)                                     # f holds no prior term, g does
        for name, sl in blocks.items():
            for _ in range(2 if name in ("M", "log_omega") else 1):
                d = np.zeros_like(x)
                d[sl] = rng.standard_normal(d[sl].size)
                d /= np.abs(d).max()
                h = 2e-5 if name == "M" else 1e-4                    # M ~ 0.15: a smaller step keeps h^2 f''' down
                fd = {}
                for hh in (h, 2 * h):
                    fd[hh] = (ev(x + hh * d)[0] - ev(x - hh * d)[0]) / (2 * hh)
                gd = g @ d
                noise = 1e2 * np.finfo(float).eps * abs(f) / h
                trunc = abs(fd[2 * h] - fd[h])
                assert abs(fd[h] - gd) < noise + trunc, (name, fd[h], gd, noise, trunc)
                assert abs(gd) > 10 * (noise + trunc), (name, gd, noise, trunc)   # the check has teeth
    finally:
        ev.close()


# ---------------------------------------------------------------- GPU: the C entries, N = 0, unsupported k, limits
@pytest.mark.gpu
def test_c_entries_match_the_lyseries_entries_with_no_lines(batch):
    import torch
    from gp_dla_detection_b200 import _lib
    lib = _lib.load()
    b = batch("k10")
    N, P, k, x = b["N"], b["P"], b["k"], b["x"]
    vp = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    out = {}
    for entry in ("gpdla_objective", "gpdla_objective_lyseries"):
        f, g = np.zeros(1), np.zeros(x.size)
        args = [N, P, k, vp(b["y"]), vp(b["lya"]), vp(b["nv"])]
        if entry.endswith("lyseries"):
            args += [0, None, None]
        _lib.check(getattr(lib, entry)(*args, vp(x), vp(f), vp(g)))
        out[entry] = f[0], g
    dev = torch.device("cuda", 0)
    t = {key: torch.from_numpy(b[key]).to(dev) for key in ("y", "lya", "nv")}
    xd = torch.from_numpy(x).to(dev)
    p = lambda a: ctypes.c_void_p(a.data_ptr())
    for entry in ("gpdla_objective_device", "gpdla_objective_lyseries_device"):
        fd = torch.zeros(1, dtype=torch.float64, device=dev)
        gd = torch.zeros(x.size, dtype=torch.float64, device=dev)
        args = [N, P, k, p(t["y"]), p(t["lya"]), p(t["nv"])]
        if entry.endswith("lyseries_device"):
            args += [0, None, None]
        _lib.check(getattr(lib, entry)(*args, p(xd), p(fd), p(gd), None))
        torch.cuda.synchronize()
        out[entry] = fd.item(), gd.cpu().numpy()
    f0, g0 = out["gpdla_objective_lyseries"]
    for entry, (f, g) in out.items():
        assert f == f0 and np.array_equal(g, g0), entry
    fr, gr = oracle_objective(b, x, "plain")
    assert_blocks(block_errors(f0, g0, fr, gr, P, k), what="gpdla_objective")


@pytest.mark.gpu
@pytest.mark.parametrize("variant", VARIANTS)
def test_no_spectra_gives_the_prior_alone(variant):
    from gp_dla_detection_b200 import api
    P, k = 333, 10
    x, y, lya, nv = OB.make_training_set(1, num_pixels=P, k=k, seed=4)
    x[-3:] += [0.2, 0.1, -0.05]
    empty = np.zeros((0, P))
    ly = lyseries_args(variant) or (0, None, None)
    f, g = api.objective_lyseries(x, empty, empty, empty, *ly)
    assert f == 0.0 and np.count_nonzero(g[:-2]) == 0
    assert np.allclose(g[-2:], prior_gradient(x)[-2:], rtol=1e-14, atol=0)
    fr, gr = OB.objective(x, empty, empty, empty, lyseries=lyseries_args(variant))
    assert fr == 0.0 and np.allclose(g, gr, rtol=1e-14, atol=0)


@pytest.mark.gpu
def test_uncompiled_rank_is_unsupported():
    from gp_dla_detection_b200 import _lib, api
    P, k = 200, 15
    x, y, lya, nv = OB.make_training_set(4, num_pixels=P, k=k, seed=6)
    with pytest.raises(_lib.GpdlaError) as err:
        api.objective(x, y, lya, nv)
    assert err.value.code == _lib.GPDLA_ERR_UNSUPPORTED and "k=15" in str(err.value)


@pytest.mark.gpu
def test_learned_optimum_belongs_to_its_x(batch):
    """learn_qso_model's reported f and gradient are those of the x it reports (against the oracle at res.x)."""
    from gp_dla_detection_b200 import api
    b = batch("k20")
    xo, fo, res = api.learn_qso_model(b["y"], b["lya"], b["nv"], b["x"], b["k"], max_iter=5)
    assert res.nit >= 1 and fo == res.fun
    fr, gr = oracle_objective(b, xo, "plain")
    e = block_errors(res.fun, res.jac, fr, gr, b["P"], b["k"])
    print("objective-scale learn_qso_model(max_iter=5) at res.x: " + " ".join("%s=%.2e" % kv for kv in e.items()))
    assert_blocks(e, what="learn_qso_model")


@pytest.mark.gpu
def test_grid_beyond_shared_memory_is_refused_as_invalid():
    """P = 12 000 at k = 40 needs ~278 KB of shared memory per CTA, more than the 227 KB a B200 block may opt in to.
    Both entries refuse it as invalid input, naming P and the largest grid that fits, before they allocate or launch
    anything, and the valid calls after it return the same bits as before."""
    from gp_dla_detection_b200 import _lib, api
    small = OB.make_training_set(300, num_pixels=200, k=40, seed=9)
    f1, g1 = api.objective(*small)
    big = OB.make_training_set(2, num_pixels=12000, k=40, seed=9)
    with pytest.raises(_lib.GpdlaError) as host_err:
        api.objective(*big)
    f2, g2 = api.objective(*small)
    assert f2 == f1 and np.array_equal(g2, g1)
    ev = api.TrainingObjective(*big[1:], 40)
    try:
        with pytest.raises(_lib.GpdlaError) as device_err:
            ev(big[0])
    finally:
        ev.close()
    f3, g3 = api.objective(*small)
    assert f3 == f1 and np.array_equal(g3, g1)
    for err in (host_err, device_err):
        assert err.value.code == _lib.GPDLA_ERR_INVALID
        assert "12000" in str(err.value) and "at most" in str(err.value)
