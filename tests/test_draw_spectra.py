"""Draws from the learned model: the NumPy restatement's random numbers against NVIDIA's Philox and its own properties on
the CPU; on the GPU the kernel against the restatement, bit reproducibility, the exact covariance of the draws, the
single-DLA catalogue calibration (asserted) and the multi-DLA one (reported)."""
import ctypes
import math
import os
import shutil
import subprocess

import numpy as np
import pytest
from scipy.stats import chi2 as chi2_dist

from gp_dla_detection_b200 import _lib, api
from gp_dla_detection_b200 import params as P
from gp_dla_detection_b200 import synthetic as syn
from oracle import draw_spectra_oracle as D
from oracle import process_qsos_oracle as O

PHILOX_HOST = r"""
#include <cstdio>
#include <cuda_runtime.h>
#define QUALIFIERS static inline __host__ __device__
#include <curand_philox4x32_x.h>
int main(int argc, char** argv) {
  FILE* in = fopen(argv[1], "rb");
  FILE* out = fopen(argv[2], "wb");
  unsigned int v[6];
  while (fread(v, sizeof v, 1, in) == 1) {
    uint4 r = curand_Philox4x32_10(make_uint4(v[0], v[1], v[2], v[3]), make_uint2(v[4], v[5]));
    unsigned int o[4] = {r.x, r.y, r.z, r.w};
    fwrite(o, sizeof o, 1, out);
  }
  fclose(in); fclose(out);
  return 0;
}
"""


def _nvcc():
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    return nvcc if os.path.exists(nvcc) else shutil.which("nvcc")


# ------------------------------------------------------------------ CPU: the oracle's random numbers
def test_oracle_philox_known_answers():
    r = D.philox4x32_10([[0, 0, 0, 0], [0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344]],
                        [[0, 0], [0xA4093822, 0x299F31D0]])
    assert [int(x) for x in r[0]] == [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]
    assert [int(x) for x in r[1]] == [0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1]


def test_oracle_philox_equals_curand(tmp_path):
    nvcc = _nvcc()
    assert nvcc, "nvcc is needed to build the library and this check"
    src = tmp_path / "philox_host.cu"
    src.write_text(PHILOX_HOST)
    exe = tmp_path / "philox_host"
    res = subprocess.run([nvcc, "-O2", "-o", str(exe), str(src)], capture_output=True, text=True)
    assert res.returncode == 0, res.stdout + res.stderr
    rng = np.random.default_rng(2024)
    v = rng.integers(0, 2 ** 32, size=(4000, 6), dtype=np.uint64).astype(np.uint32)
    v[:8, :4] = 0                                  # small counters as the kernel uses them
    v[8:16, 4:] = 0xFFFFFFFF                       # keys that wrap in the Weyl sequence
    (tmp_path / "in.bin").write_bytes(v.tobytes())
    subprocess.run([str(exe), str(tmp_path / "in.bin"), str(tmp_path / "out.bin")], check=True)
    want = np.frombuffer((tmp_path / "out.bin").read_bytes(), dtype=np.uint32).reshape(-1, 4)
    got = D.philox4x32_10(v[:, :4].astype(np.uint64), v[:, 4:].astype(np.uint64)).astype(np.uint32)
    assert want.shape == got.shape == (4000, 4)
    assert np.array_equal(got, want)


def test_oracle_uniforms_and_indices_in_range():
    w0, w1 = D.words(12345, np.arange(20000), D.STREAM_PIXEL, 7)
    u = np.concatenate([D.uniform(w0), D.uniform(w1)])
    assert np.all(u > 0.0) and np.all(u < 1.0)
    assert abs(u.mean() - 0.5) < 4 * math.sqrt(1 / 12 / u.size)
    for S in (1, 7, 10000, 2 ** 31 - 1):
        i = D.umulhi64(w0, S)
        assert i.min() >= 0 and i.max() < S
    assert np.array_equal(D.umulhi64(np.array([2 ** 64 - 1, 2 ** 63, 12345], dtype=np.uint64), 10000),
                          np.array([((2 ** 64 - 1) * 10000) >> 64, (2 ** 63 * 10000) >> 64, (12345 * 10000) >> 64],
                                   dtype=np.uint64))
    a, b = D.normals(w0, w1)
    n = np.concatenate([a, b])
    assert abs(n.mean()) < 4 / math.sqrt(n.size) and abs(n.var() - 1) < 4 * math.sqrt(2 / n.size)


def _multi_prior(dla_fraction, n=20000, seed=3):
    rng = np.random.default_rng(seed)
    return dict(z_qsos=rng.uniform(2.0, 5.0, n), dla_ind=(rng.random(n) < dla_fraction).astype(np.uint8))


@pytest.mark.parametrize("kind", [0, 1])
def test_oracle_model_frequencies_follow_the_priors(kind):
    prior = _multi_prior(0.4)
    p = D.model_probabilities(prior, 3.0, kind, 4, 0.18, 0.82)
    assert abs(p.sum() - 1) < 1e-12
    Qn = 100000
    u = D.uniform(D.words(99, np.arange(Qn), D.STREAM_MODEL, 0)[0])
    m = np.array([D.choose_model(p, x)[0] for x in u[:2000]])
    edges = np.cumsum(p)
    fast = np.minimum(np.searchsorted(edges, u, side="right"), p.size - 1)
    assert np.array_equal(m, fast[:2000])
    counts = np.bincount(fast, minlength=p.size)
    stat = np.sum((counts - Qn * p) ** 2 / (Qn * p))
    assert chi2_dist.sf(stat, p.size - 1) > 1e-4, (counts, Qn * p)


def test_oracle_separation_and_truth_z_bits():
    off = syn.make_samples(10000)["offset_samples"]
    sep = D.MIN_Z_SEPARATION
    accepted = 0
    lo, hi = 2.2, 2.2 + 40 * sep                     # 4 DLAs in a short range: many sets are rejected
    for g in range(400):
        got = D.draw_absorbers(7, g, 5, off.size, lo, hi, off)
        if got is None:
            continue
        ind, z = got
        accepted += 1
        assert np.all(np.diff(z) >= sep)
        assert np.array_equal(z, lo + (hi - lo) * off[ind])
        assert np.all((ind >= 0) & (ind < off.size))
    assert accepted > 100
    # truth z of full draws: min_z + span * offset[i] with the used-pixel range, bit for bit
    model, samples = syn.make_model(), syn.make_samples(10000, with_lls=True)
    prior = _multi_prior(0.6)
    sp = syn.make_spectra(model, 40, seed=5)
    res = D.draw_spectra(model, samples, prior, sp, seed=3, kind=1, max_dlas=4, Z_lls=0.18, Z_dla=0.82)
    seen = 0
    for q in range(40):
        code = res["truth_model"][q]
        if code < 1:
            continue
        lam, zq = sp["all_wavelengths"][q], sp["z_qsos"][q]
        rest = lam / (1 + zq)
        used = lam[(rest >= O.min_lambda) & (rest <= O.max_lambda) & ~np.asarray(sp["all_pixel_mask"][q], bool)]
        lo, hi = O.min_z_dla(used, zq), O.max_z_dla(used, zq)
        j = 1 if code == 1 else code - 1
        ind = res["truth_inds"][q, :j]
        assert np.array_equal(res["truth_z"][q, :j], lo + (hi - lo) * samples["offset_samples"][ind])
        assert np.all(np.diff(res["truth_z"][q, :j]) >= D.MIN_Z_SEPARATION)
        assert np.all(res["truth_inds"][q, j:] == -1) and np.all(np.isnan(res["truth_z"][q, j:]))
        want = np.log10(samples["lls_nhi_samples"][ind]) if code == 1 else samples["log_nhi_samples"][ind]
        assert np.array_equal(res["truth_log_nhi"][q, :j], want)
        seen += 1
    assert seen > 10


def test_oracle_short_window_flags_unseparated_sets():
    model, samples = syn.make_model(), syn.make_samples(1000, with_lls=True)
    sp = syn.make_spectra(model, 1, seed=9)
    lam, zq = sp["all_wavelengths"][0], float(sp["z_qsos"][0])
    rest = lam / (1 + zq)
    win = np.nonzero((rest >= O.min_lambda) & (rest <= O.max_lambda))[0]
    keep = win[:4]                   # 4 window pixels: |max_z - min_z| is about kms_to_z(3000), too short for 3 DLAs
    short = dict(all_wavelengths=[lam[keep]] * 60, all_flux=[sp["all_flux"][0][keep]] * 60,
                 all_noise_variance=[sp["all_noise_variance"][0][keep]] * 60,
                 all_pixel_mask=[np.zeros(4, bool)] * 60, z_qsos=np.full(60, zq))
    res = D.draw_spectra(model, samples, _multi_prior(0.8), short, seed=1, kind=1, max_dlas=4, Z_lls=0.18, Z_dla=0.82)
    codes = res["truth_model"]
    assert np.any(codes == -2) and not np.any(codes >= 4)
    assert np.all(np.isnan(res["flux"][codes == -2]))
    assert np.all(np.isfinite(res["flux"][codes >= 0]))


# ------------------------------------------------------------------ GPU
def _up(a, dt):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, dtype=dt)).cuda()


def _planes(pad):
    return (_up(pad["wavelengths"], np.float64), _up(pad["flux"], np.float64), _up(pad["noise_variance"], np.float64),
            _up(pad["pixel_mask"], np.uint8), _up(pad["lengths"], np.int32), _up(pad["z_qsos"], np.float64))


def _spectra(model, Q, seed, meanflux=False):
    """make_spectra setups plus a quasar whose window is all masked and one with no window pixel."""
    sp = syn.make_spectra(model, Q, seed=seed, dla_fraction=0.3, meanflux=meanflux)
    lam, z = sp["all_wavelengths"][0], sp["z_qsos"][0]
    rest = lam / (1 + z)
    win = (rest >= P.DEFAULT.min_lambda) & (rest <= P.DEFAULT.max_lambda)
    for w, f, v, m in ((lam, sp["all_flux"][0], sp["all_noise_variance"][0], win | sp["all_pixel_mask"][0]),
                       (lam[:5], sp["all_flux"][0][:5], sp["all_noise_variance"][0][:5], np.zeros(5, bool))):
        sp["all_wavelengths"].append(w); sp["all_flux"].append(f); sp["all_noise_variance"].append(v)
        sp["all_pixel_mask"].append(m)
        sp["z_qsos"] = np.append(sp["z_qsos"], z)
    return sp


def _given(sp, rng, A=4):
    """0..A absorbers per quasar inside its window, separated, N in [10^19.5, 10^22]."""
    Q = len(sp["z_qsos"])
    z, n = np.full((Q, A), np.nan), np.full((Q, A), np.nan)
    for q in range(Q):
        lam, zq = sp["all_wavelengths"][q], sp["z_qsos"][q]
        rest = lam / (1 + zq)
        w = lam[(rest >= P.DEFAULT.min_lambda) & (rest <= P.DEFAULT.max_lambda)]
        if w.size == 0:
            continue
        lo, hi = w.min() / P.lya_wavelength - 1, w.max() / P.lya_wavelength - 1
        m = q % (A + 1)
        z[q, :m] = np.sort(rng.uniform(lo, hi, m))
        n[q, :m] = 10.0 ** rng.uniform(19.5, 22.0, m)
    return z, n


def _processor(k=20, S=10000, prior=None):
    return api.DLAProcessor(syn.make_model(k), syn.make_samples(S, with_lls=True), prior or syn.make_prior(), device=0)


def _compare(got, ref, scale, label):
    """truth bit-equal except choices within 1e-12 of a cumulative edge (counted); flux within 1e-12 scale."""
    near = ref["edge"] < 1e-12
    ok = ~near
    if "truth_model" in got:
        for nm in ("truth_model", "truth_inds", "truth_z", "truth_log_nhi"):
            assert np.array_equal(got[nm][ok], ref[nm][ok], equal_nan=True), (label, nm)
    rows = ok & (np.isfinite(got["flux"]).any(axis=1) | np.isfinite(ref["flux"]).any(axis=1))
    g, r = got["flux"][rows], ref["flux"][rows]
    assert np.array_equal(np.isnan(g), np.isnan(r)), label
    fin = np.isfinite(r)
    sc = scale[rows]
    sc = np.where(np.isfinite(sc), sc, 1.0)           # outside the window: copied, so equal
    err = np.abs(g[fin] - r[fin]) / sc[fin]
    assert err.max(initial=0.0) <= 1e-12, (label, err.max())
    print("%s: %d quasars, max flux error %.2e of the pixel scale, %d model choices near an edge"
          % (label, rows.sum(), err.max(initial=0.0), near.sum()))


@pytest.mark.gpu
@pytest.mark.parametrize("k", [10, 20, 40])
def test_kernel_matches_oracle(k):
    model = syn.make_model(k)
    samples = syn.make_samples(10000, with_lls=True)
    prior = syn.make_prior()
    Q = 300 if k == 20 else 60
    sp = _spectra(model, Q, seed=40 + k)
    pad = api.pad_spectra(sp)
    L_max = pad["flux"].shape[1]
    az, an = _given(sp, np.random.default_rng(k))
    proc = api.DLAProcessor(model, samples, prior, device=0)
    try:
        # the pixel scale |prior_mean| + prior_sd, with every window pixel unmasked so that prior_sd is defined
        unmasked = dict(pad, pixel_mask=np.zeros_like(pad["pixel_mask"]))
        cases = [("draw prior single", dict(model="single"), {}),
                 ("draw prior multi", dict(model="multi", max_dlas=4), {}),
                 ("draw given single", dict(model="single", absorber_z=az, absorber_nhi=an), {}),
                 ("draw given multi", dict(model="multi", absorber_z=az, absorber_nhi=an), {}),
                 ("inject prior single", dict(model="single", inject=True), {}),
                 ("inject given multi", dict(model="multi", inject=True, absorber_z=az, absorber_nhi=an), {})]
        if k != 20:
            cases = [cases[1], cases[5]]
        for label, kw, _ in cases:
            got = proc.draw_spectra(pad, seed=1000 + k, first_quasar=17, **kw)
            kind = int(kw["model"] == "multi")
            ref = D.draw_spectra(model, samples, prior, sp, 1000 + k, first_quasar=17, kind=kind,
                                 max_dlas=kw.get("max_dlas", 4), inject=kw.get("inject", False),
                                 absorber_z=kw.get("absorber_z"), absorber_nhi=kw.get("absorber_nhi"),
                                 num_lines=proc.params.num_lines, L_max=L_max, Z_lls=samples["Z_lls"],
                                 Z_dla=samples["Z_dla"])
            if "truth_inds" in got:
                rz, rn = api.truth_absorbers(got, samples)
            else:
                rz, rn = kw["absorber_z"], kw["absorber_nhi"]
            rec = proc.reconstruct(unmasked, rz, rn, meanflux=bool(kind))
            scale = np.abs(rec["prior_mean"]) + rec["prior_sd"]
            if kw.get("inject"):
                scale = scale + np.abs(pad["flux"])
            _compare(got, ref, scale, "k=%d %s" % (k, label))
            # the absorption is reconstruct's plane for the same absorbers, bit for bit
            rec_abs = proc.reconstruct(pad, rz, rn, meanflux=bool(kind))["absorption"]
            drawn = got["truth_model"] >= 0 if "truth_model" in got else np.ones(len(rec_abs), bool)
            assert np.array_equal(got["absorption"][drawn], rec_abs[drawn], equal_nan=True), label
            if "truth_z" in got and not kw.get("inject"):
                # the truth z is the z processing assigns to the sample, on the drawn batch
                out = proc.process_device(*_planes(got))
                zlo, zhi = out["min_z_dlas"].cpu().numpy(), out["max_z_dlas"].cpu().numpy()
                ind = got["truth_inds"]
                on = ind >= 0
                want = zlo[:, None] + (zhi - zlo)[:, None] * samples["offset_samples"][np.where(on, ind, 0)]
                assert np.array_equal(got["truth_z"][on], want[on]), label
    finally:
        proc.close()


@pytest.mark.gpu
def test_bits_repeat_host_device_halves_and_empty_injection():
    import torch
    model = syn.make_model()
    sp = _spectra(model, 40, seed=8)
    pad = api.pad_spectra(sp)
    proc = _processor()
    try:
        for kw in (dict(model="multi"), dict(model="single", inject=True)):
            a = proc.draw_spectra(pad, seed=5, **kw)
            b = proc.draw_spectra(pad, seed=5, **kw)
            W, F, V, Mk, Ln, Z = _planes(pad)
            dev = proc.draw_spectra_device(W, F, V, Mk, Ln, Z, seed=5, **kw)
            torch.cuda.synchronize()
            for nm in dev:
                assert np.array_equal(a[nm], b[nm], equal_nan=True), nm
                assert np.array_equal(a[nm], dev[nm].cpu().numpy(), equal_nan=True), nm
            h = 17
            halves = [proc.draw_spectra_device(W[s], F[s], V[s], Mk[s], Ln[s], Z[s], seed=5, first_quasar=f, **kw)
                      for s, f in ((slice(0, h), 0), (slice(h, None), h))]
            for nm in dev:
                whole = torch.cat([halves[0][nm], halves[1][nm]]).cpu().numpy()
                assert np.array_equal(whole, a[nm], equal_nan=True), nm
            assert not np.array_equal(proc.draw_spectra(pad, seed=6, **kw)["flux"], a["flux"], equal_nan=True)
        Q = pad["flux"].shape[0]
        same = proc.draw_spectra(pad, seed=5, inject=True, absorber_z=np.zeros((Q, 0)), absorber_nhi=np.zeros((Q, 0)))
        live = np.isfinite(same["absorption"]).any(axis=1)
        assert live.sum() == Q - 2
        assert np.array_equal(same["flux"][live], pad["flux"][live])
    finally:
        proc.close()


@pytest.mark.gpu
def test_argument_checks():
    lib = _lib.load()
    proc = _processor(S=100)
    sp = api.pad_spectra(syn.make_spectra(syn.make_model(), 2, seed=1))
    try:
        vp = lambda a: ctypes.c_void_p(np.ascontiguousarray(a).ctypes.data)
        W, F, V = (np.ascontiguousarray(sp[k]) for k in ("wavelengths", "flux", "noise_variance"))
        Mk, Ln, Z = (np.ascontiguousarray(sp["pixel_mask"], dtype=np.uint8),
                     np.ascontiguousarray(sp["lengths"], dtype=np.int32), np.ascontiguousarray(sp["z_qsos"]))
        flux = np.empty_like(W)
        tm, ti, tz, tn = np.empty(2, np.int32), np.empty(2, np.int64), np.empty(2), np.empty(2)
        az = np.full((2, 1), 2.5)

        def call(ctx, fin=True, truth=True, **opt):
            o = _lib.GpdlaDrawOptions()
            o.model, o.max_dlas, o.from_prior = 0, 1, 1
            for key, val in opt.items():
                setattr(o, key, val)
            out = _lib.GpdlaDrawOutputs()
            out.flux = flux.ctypes.data
            if truth:
                out.truth_model, out.truth_inds, out.truth_z, out.truth_log_nhi = (
                    tm.ctypes.data, ti.ctypes.data, tz.ctypes.data, tn.ctypes.data)
            return lib.gpdla_draw_spectra(ctx, 2, W.shape[1], vp(W), vp(F) if fin else None, vp(V), vp(Mk), vp(Ln),
                                          vp(Z), ctypes.byref(o), ctypes.byref(out))
        assert call(proc._ctx) == _lib.GPDLA_OK
        assert call(proc._ctx, fin=False, inject=1) == _lib.GPDLA_ERR_INVALID
        assert call(proc._ctx, num_absorbers=1, absorber_z=az.ctypes.data,
                    absorber_nhi=az.ctypes.data) == _lib.GPDLA_ERR_INVALID
        assert call(proc._ctx, first_quasar=-1) == _lib.GPDLA_ERR_INVALID
        assert call(proc._ctx, truth=False) == _lib.GPDLA_ERR_INVALID
        assert call(proc._ctx, model=1, max_dlas=5) == _lib.GPDLA_ERR_INVALID
        assert call(proc._ctx, model=2) == _lib.GPDLA_ERR_INVALID
        empty = ctypes.c_void_p()
        _lib.check(lib.gpdla_create(ctypes.byref(empty), 0))
        try:
            assert call(empty) == _lib.GPDLA_ERR_STATE
            assert call(empty, fin=False, inject=1) == _lib.GPDLA_ERR_INVALID   # argument checks come first
        finally:
            lib.gpdla_destroy(empty)
        no_lls = api.DLAProcessor(syn.make_model(), syn.make_samples(100), syn.make_prior(2000), device=0)
        try:
            assert call(no_lls._ctx, model=1, max_dlas=2) == _lib.GPDLA_ERR_STATE
            assert call(no_lls._ctx, model=0) == _lib.GPDLA_OK
        finally:
            no_lls.close()
    finally:
        proc.close()


def _chi2_check(chi2, n):
    ok = np.isfinite(chi2) & (n > 0)
    chi2, n = chi2[ok], n[ok].astype(np.float64)
    t = (chi2 - n) / np.sqrt(2 * n)
    total = abs(chi2.sum() - n.sum()) <= 5 * math.sqrt(2 * n.sum())
    return total and abs(t.var() - 1) <= 0.15, (chi2.sum() - n.sum()) / math.sqrt(2 * n.sum()), t.var()


@pytest.mark.gpu
def test_draws_follow_the_model_covariance_exactly():
    model = syn.make_model()
    Q = 2000
    sp = syn.make_spectra(model, Q, seed=21)
    pad = api.pad_spectra(sp)
    az, an = _given(sp, np.random.default_rng(4), A=3)
    an = np.where(np.isnan(az), np.nan, np.maximum(an, 10.0 ** 20.5))
    proc = _processor()
    try:
        planes = _planes(pad)
        W, F, V, Mk, Ln, Z = planes

        def chi2_of(flux, z, n, meanflux):
            r = proc.reconstruct_device(W, flux, V, Mk, Ln, Z, absorber_z=z, absorber_nhi=n, meanflux=meanflux)
            return r["chi2"].cpu().numpy(), r["num_pixels"].cpu().numpy()

        rows = {}
        single = proc.draw_spectra_device(*planes, seed=11, absorber_z=az, absorber_nhi=an)["flux"]
        rows["draw, single-DLA null model"] = (_chi2_check(*chi2_of(single, az, an, False)), True)
        null = proc.draw_spectra_device(*planes, seed=12, absorber_z=np.zeros((Q, 0)), absorber_nhi=np.zeros((Q, 0)))
        inj = proc.draw_spectra_device(W, null["flux"], V, Mk, Ln, Z, seed=13, inject=True, absorber_z=az,
                                       absorber_nhi=an)["flux"]
        rows["inject on a null draw"] = (_chi2_check(*chi2_of(inj, az, an, False)), True)
        mf = proc.draw_spectra_device(*planes, seed=14, model="multi", absorber_z=az, absorber_nhi=an)["flux"]
        rows["draw, mean-flux null model"] = (_chi2_check(*chi2_of(mf, az, an, True)), True)
        rows["control: absorbers dropped"] = (_chi2_check(*chi2_of(single, None, None, False)), False)
        rows["control: the other null model"] = (_chi2_check(*chi2_of(single, az, an, True)), False)
        for label, ((passed, z, var), want) in rows.items():
            print("%-32s (sum chi2 - sum n) / sqrt(2 sum n) = %8.2f, var = %.3f" % (label, z, var))
            assert passed == want, label
    finally:
        proc.close()


@pytest.mark.gpu
def test_single_dla_catalogue_calibration():
    from test_dla_posteriors import _coverage_check
    import torch
    model = syn.make_model()
    samples = syn.make_samples(10000)
    Q, probs = 4000, tuple(np.round(np.arange(1, 10) / 10.0, 1))
    sp = syn.make_spectra(model, Q, seed=33)
    pad = api.pad_spectra(sp)
    proc = api.DLAProcessor(model, samples, syn.make_prior(), device=0)
    try:
        W, F, V, Mk, Ln, Z = _planes(pad)
        draw = proc.draw_spectra_device(W, F, V, Mk, Ln, Z, seed=2024)
        out = proc.process_device(W, draw["flux"], V, Mk, Ln, Z, return_sample_log_likelihoods=True)
        truth = {k: v.cpu().numpy() for k, v in draw.items() if k.startswith("truth")}
        valid = truth["truth_model"] >= 0
        sel = torch.from_numpy(valid.astype(np.uint8)).cuda()
        lnhi = samples["log_nhi_samples"]
        nhi_edges = np.array([lnhi.min() - 1e-9, *np.quantile(lnhi, [1 / 3, 2 / 3]), lnhi.max() + 1e-9])
        z_edges = np.array([0.0, 10.0])
        stats = api.unpack_dla_statistics(proc.statistics_device(out, z_edges, nhi_edges, select=sel), 1, 3)
        rec = proc.posteriors_device(out, quantiles=probs).cpu().numpy()
        p_dla = out["p_dlas"].cpu().numpy()
        ll = out["sample_log_likelihoods_dla"].cpu().numpy()
    finally:
        proc.close()
    assert np.all(truth["truth_model"] >= -1) and valid.sum() > 0.95 * Q
    dla = truth["truth_model"] == 2
    p = p_dla[valid]
    n_dla, expect, sd = dla.sum(), p.sum(), math.sqrt(np.sum(p * (1 - p)))
    print("single-DLA catalogue: %d drawn DLAs, sum p_dla = %.1f +- %.1f" % (n_dla, expect, sd))
    assert abs(n_dla - expect) <= 4 * sd
    tz, tn = truth["truth_z"][:, 0], truth["truth_log_nhi"][:, 0]
    for c in range(3):
        drawn = np.count_nonzero(dla & (tn >= nhi_edges[c]) & (tn < nhi_edges[c + 1]))
        e, v = stats["counts"][0, c], stats["counts_var"][0, c]
        print("cell log N [%.2f, %.2f): drawn %d, expected %.1f +- %.1f" % (nhi_edges[c], nhi_edges[c + 1], drawn, e,
                                                                         math.sqrt(v)))
        assert abs(drawn - e) <= 4 * math.sqrt(v)
    t = api.unpack_dla_posteriors(rec[dla], len(probs))
    w = np.exp(ll[dla] - ll[dla].max(axis=1, keepdims=True))
    w_max = 1.0 / w.sum(axis=1)
    perm = np.random.default_rng(5).permutation(dla.sum())
    for name, truths, qv in (("z", tz[dla], t["z_quantiles"]), ("log N", tn[dla], t["log_nhi_quantiles"])):
        rows = _coverage_check(truths, qv, probs, w_max)
        control = _coverage_check(truths[perm], qv, probs, w_max)
        for (pp, n, lo, hi, ok), (_, nc, _, _, okc) in zip(rows, control):
            print("coverage %-5s p = %.1f: %4d truths <= q_p, allowed [%.1f, %.1f]; permuted control %4d%s"
                  % (name, pp, n, lo, hi, nc, "" if okc else " (outside)"))
        assert all(r[4] for r in rows), name
        assert not all(r[4] for r in control), name + ": the permuted control passes the check"


@pytest.mark.gpu
def test_multi_dla_catalogue_reported():
    import torch
    model = syn.make_model()
    samples = syn.make_samples(10000, with_lls=True)
    Q, J = 2000, 4
    sp = syn.make_spectra(model, Q, seed=34, meanflux=True)
    pad = api.pad_spectra(sp)
    proc = api.DLAProcessor(model, samples, syn.make_prior(), device=0)
    try:
        planes = _planes(pad)
        W, F, V, Mk, Ln, Z = planes
        draw = proc.draw_spectra_device(*planes, seed=77, model="multi", max_dlas=J)
        out = proc.process_multi_device(W, draw["flux"], V, Mk, Ln, Z, max_dlas=J, return_samples=True)
        probs = (0.16, 0.5, 0.84)
        qrec = api.unpack_multi_dla_posterior_quantiles(proc.multi_posterior_quantiles_device(out, quantiles=probs),
                                                        J, len(probs))
        mp = out["model_posteriors"].cpu().numpy()
        zlo, zhi = out["min_z_dlas"].cpu().numpy(), out["max_z_dlas"].cpu().numpy()
        truth = {k: v.cpu().numpy() for k, v in draw.items() if k.startswith("truth")}
        flux = draw["flux"].cpu().numpy()
        # given 2- and 3-absorber sets
        rng = np.random.default_rng(8)
        gz, gn = np.full((Q, 3), np.nan), np.full((Q, 3), np.nan)
        for q in range(Q):
            if not np.isfinite(zlo[q]) or zhi[q] - zlo[q] < 0.1:
                continue
            m = 2 + q % 2
            gz[q, :m] = zlo[q] + (zhi[q] - zlo[q]) * (np.arange(m) + rng.uniform(0.2, 0.8, m)) / m
            gn[q, :m] = 10.0 ** rng.uniform(20.3, 21.5, m)
        given = proc.draw_spectra_device(*planes, seed=78, model="multi", absorber_z=gz, absorber_nhi=gn)
        gout = proc.process_multi_device(W, given["flux"], V, Mk, Ln, Z, max_dlas=J)
        gmp = gout["model_posteriors"].cpu().numpy()
    finally:
        proc.close()
    codes = truth["truth_model"]
    ok = codes >= 0
    # sanity, asserted: finite window flux outside flagged rows, separated sets, the z-range bits
    W_h, L_h = pad["wavelengths"], pad["lengths"]
    rest = W_h / (1 + pad["z_qsos"][:, None])
    win = (rest >= P.DEFAULT.min_lambda) & (rest <= P.DEFAULT.max_lambda) & (np.arange(W_h.shape[1]) < L_h[:, None])
    assert np.all(np.isfinite(flux[ok][win[ok]]))
    assert np.all(np.isnan(flux[~ok]))
    for q in np.nonzero(codes >= 3)[0]:
        assert np.all(np.diff(truth["truth_z"][q, :codes[q] - 1]) >= D.MIN_Z_SEPARATION)
    on = truth["truth_inds"] >= 0
    want = zlo[:, None] + (zhi - zlo)[:, None] * samples["offset_samples"][np.where(on, truth["truth_inds"], 0)]
    assert np.array_equal(truth["truth_z"][on], want[on])
    # reported: the evidence is importance-sampled, so this calibration is close to, not exactly, an identity
    fin = ok & np.all(np.isfinite(mp), axis=1)
    names = ["no DLA", "sub-DLA"] + ["%d DLA" % j for j in range(1, J + 1)]
    print("multi-DLA prior draws: %d quasars, %d flagged (-2), %d without a draw (-1)"
          % (Q, np.sum(codes == -2), np.sum(codes == -1)))
    for m, nm in enumerate(names):
        print("  %-8s drawn %4d, sum of model posteriors %8.1f" % (nm, np.sum(codes[fin] == m), mp[fin, m].sum()))
    two = fin & (codes == 3)
    if two.any():
        zq = qrec["z_quantiles"][two, 1, :2]              # level 2, ranks 0 and 1; quantiles (0.16, 0.5, 0.84)
        tz = truth["truth_z"][two, :2]
        inside = (tz >= zq[:, :, 0]) & (tz <= zq[:, :, 2])
        print("  level-2 68 %% z interval coverage over %d two-DLA quasars: rank 0 %.2f, rank 1 %.2f"
              % (two.sum(), inside[:, 0].mean(), inside[:, 1].mean()))
    gcount = np.sum(np.isfinite(gz), axis=1)
    for m in (2, 3):
        s = (gcount == m) & np.all(np.isfinite(gmp), axis=1)
        print("  given %d DLAs: %d quasars, mean posterior of %d DLAs %.3f, of the MAP model being it %.3f"
              % (m, s.sum(), m, gmp[s, 1 + m].mean(), np.mean(np.argmax(gmp[s], axis=1) == 1 + m)))
