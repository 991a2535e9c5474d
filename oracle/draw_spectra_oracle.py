"""Literal CPU restatement of the draws from the learned model (test oracle for ``gpdla_draw_spectra``).

TEST INFRASTRUCTURE ONLY -- see ``oracle/__init__.py``.  parity unpinned: the reference has no generative entry point;
the model being sampled is the one its inference evaluates (process_qsos.m, ...meanflux.m), and the random-number layout
is the library's own (include/gpdla.h, gpdla_draw_spectra).  Uses none of the kernel's code: Philox4x32-10 in uint64
NumPy arithmetic, the absorption from this package's ``voigt`` / ``padded_wavelengths``, the null model from
``reconstruct_oracle.window_model``, the priors from ``process_qsos_oracle.log_priors`` and
``process_qsos_multi_oracle.multi_priors``.

Per quasar, on the modelled window (masked pixels included), with a the product of the absorbers' convolved profiles:
  draw    y = a (mu~ + M~ xi + om2~^(1/2) e1) + v^(1/2) e2           (NaN outside the window, 0 past the length)
  inject  y' = a y + ((1 - a^2) v)^(1/2) e2, the noise term 0 where a^2 >= 1   (other pixels copied)
Random words: Philox4x32-10 with key = seed, counter = (element, stream, g_lo, g_hi), g = first_quasar + q;
W0 = r1:r0, W1 = r3:r2.  Stream 0 element 0: model choice u = ((W0 >> 11) + 0.5) 2^-53; stream 1 element
4 attempt + slot: sample index umulhi64(W0, S); stream 2 element c: xi_2c, xi_2c+1; stream 3 element i: e1, e2 of
pixel i; normals by Box-Muller r = sqrt(-2 log u0), (r cos(pi 2u1), r sin(pi 2u1)).
"""
from __future__ import annotations

import math

import numpy as np

from . import process_qsos_multi_oracle as MO
from . import process_qsos_oracle as O
from . import reconstruct_oracle as R

MASK32 = np.uint64(0xFFFFFFFF)
PHILOX_M0, PHILOX_M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
PHILOX_W0, PHILOX_W1 = np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)
STREAM_MODEL, STREAM_INDEX, STREAM_LATENT, STREAM_PIXEL = 0, 1, 2, 3
MAX_ATTEMPTS = 64
MIN_Z_SEPARATION = O.kms_to_z(3000.0)       # ...meanflux.m:33


def philox4x32_10(counter, key):
    """Philox4x32-10 (Salmon et al. 2011) on arrays: counter [..., 4], key [..., 2] of 32-bit words -> [..., 4]."""
    c = [np.asarray(counter, dtype=np.uint64)[..., i] & MASK32 for i in range(4)]
    k = [np.asarray(key, dtype=np.uint64)[..., i] & MASK32 for i in range(2)]
    for r in range(10):
        if r:
            k = [(k[0] + PHILOX_W0) & MASK32, (k[1] + PHILOX_W1) & MASK32]
        p0, p1 = PHILOX_M0 * c[0], PHILOX_M1 * c[2]                  # < 2^64: exact in uint64
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k[0], p1 & MASK32, (p0 >> np.uint64(32)) ^ c[3] ^ k[1], p0 & MASK32]
    return np.stack(c, axis=-1)


def words(seed, g, stream, element):
    """(W0, W1) uint64 of the draws at (seed, g, stream, element); g and element may be arrays (broadcast)."""
    element, g = np.broadcast_arrays(np.atleast_1d(np.asarray(element, dtype=np.uint64)), np.asarray(g, dtype=np.uint64))
    seed = int(seed) & (2 ** 64 - 1)
    ctr = np.stack([element, np.full_like(element, stream), g & MASK32, g >> np.uint64(32)], axis=-1)
    key = np.broadcast_to(np.array([seed & 0xFFFFFFFF, seed >> 32], dtype=np.uint64), ctr.shape[:-1] + (2,))
    r = philox4x32_10(ctr, key)
    return (r[..., 1] << np.uint64(32)) | r[..., 0], (r[..., 3] << np.uint64(32)) | r[..., 2]


def uniform(w):
    """((W >> 11) + 0.5) 2^-53"""
    return ((np.asarray(w, dtype=np.uint64) >> np.uint64(11)).astype(np.float64) + 0.5) * 2.0 ** -53


def umulhi64(a, b):
    """The high 64 bits of the 128-bit product of two uint64 values."""
    a, b = np.asarray(a, dtype=np.uint64), np.uint64(b)
    a_lo, a_hi, b_lo, b_hi = a & MASK32, a >> np.uint64(32), b & MASK32, b >> np.uint64(32)
    ll, lh, hl, hh = a_lo * b_lo, a_lo * b_hi, a_hi * b_lo, a_hi * b_hi
    mid = (ll >> np.uint64(32)) + (lh & MASK32) + (hl & MASK32)
    return hh + (lh >> np.uint64(32)) + (hl >> np.uint64(32)) + (mid >> np.uint64(32))


def normals(w0, w1):
    r = np.sqrt(-2.0 * np.log(uniform(w0)))
    t = 2.0 * uniform(w1)
    return r * np.cos(np.pi * t), r * np.sin(np.pi * t)


def model_probabilities(prior, z_qso, kind, max_dlas, Z_lls=None, Z_dla=None):
    """The model probabilities in truth-code order: single (none, 1 DLA); multi (none, sub-DLA, 1..J DLAs)."""
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        if kind == 0:
            lp = np.array(O.log_priors(prior["z_qsos"], prior["dla_ind"], z_qso))
        else:
            no, lls, dla = MO.multi_priors(prior["z_qsos"], prior["dla_ind"], z_qso, max_dlas, Z_lls, Z_dla)
            lp = np.concatenate([[no, lls], dla])
        return np.exp(lp)


def choose_model(p, u):
    """The first m with u < sum_{<= m} p (running sum in order), else the last; and u's distance to the nearest edge."""
    edges, cum = [], 0.0
    for t in range(len(p)):
        cum = cum + p[t]
        edges.append(cum)
    m = next((t for t, e in enumerate(edges) if u < e), len(p) - 1)
    return m, float(np.min(np.abs(np.asarray(edges) - u)))


def draw_absorbers(seed, g, code, S, min_z, max_z, offsets):
    """Sample indices and z of `code`'s absorbers (1: one sub-DLA sample, 1 + j: j separated DLA samples), ascending z;
    None if 64 attempts find no separated set."""
    j = 1 if code == 1 else code - 1
    span = max_z - min_z
    for att in range(MAX_ATTEMPTS):
        w0, _ = words(seed, g, STREAM_INDEX, 4 * att + np.arange(j))
        ind = umulhi64(w0, S).astype(np.int64)
        z = min_z + span * offsets[ind]
        order = np.argsort(z, kind="stable")
        ind, z = ind[order], z[order]
        if not np.any(np.diff(z) < MIN_Z_SEPARATION):
            return ind, z
    return None


def draw_one(model, samples, prior, wavelengths, flux, noise_variance, pixel_mask, z_qso, seed, g, kind=0,
             max_dlas=4, inject=False, absorber_z=(), absorber_nhi=(), from_prior=True, num_lines=O.num_lines_default,
             Z_lls=None, Z_dla=None):
    """One quasar's row (its own pixels): flux and absorption (None for a NaN row: no used pixel or no draw), the truth
    (code, indices, z, log N) of a prior draw, and its model choice's distance to the nearest cumulative edge (inf when
    no choice was made)."""
    wl = np.asarray(wavelengths, dtype=np.float64)
    y_in = np.asarray(flux, dtype=np.float64)
    v = np.asarray(noise_variance, dtype=np.float64)
    mask = np.asarray(pixel_mask).astype(bool)
    L = wl.size
    rest = wl / (1.0 + z_qso)
    win = (rest >= O.min_lambda) & (rest <= O.max_lambda)
    used = win & ~mask
    TW = max_dlas if kind == 1 else 1
    truth = dict(code=0, inds=np.full(TW, -1, np.int64), z=np.full(TW, np.nan), log_nhi=np.full(TW, np.nan))
    edge = math.inf
    if from_prior:
        p = model_probabilities(prior, z_qso, kind, max_dlas, Z_lls, Z_dla)
        if not np.any(used) or not np.all(np.isfinite(p)):
            truth["code"] = -1
            return None, truth, edge
        w0, _ = words(seed, g, STREAM_MODEL, 0)
        m, edge = choose_model(p, float(uniform(w0)[0]))
        code = 2 if (kind == 0 and m == 1) else m
        truth["code"] = code
        az, an = [], []
        if code > 0:
            lam = wl[used]
            min_z, max_z = O.min_z_dla(lam, z_qso), O.max_z_dla(lam, z_qso)
            got = draw_absorbers(seed, g, code, samples["offset_samples"].size, min_z, max_z,
                                 samples["offset_samples"])
            if got is None:
                truth["code"] = -2
                return None, truth, edge
            ind, zz = got
            n = samples["lls_nhi_samples"][ind] if code == 1 else samples["nhi_samples"][ind]
            truth["inds"][:ind.size], truth["z"][:ind.size] = ind, zz
            truth["log_nhi"][:ind.size] = np.log10(n) if code == 1 else samples["log_nhi_samples"][ind]
            az, an = zz, n
    else:
        az, an = np.ravel(absorber_z), np.ravel(absorber_nhi)
        if not np.any(used):
            return None, truth, edge
    w_win = wl[win]
    absorption = np.ones(w_win.size)
    padded = O.padded_wavelengths(w_win)
    for z, N in zip(az, an):
        if np.isnan(z):
            continue
        absorption = absorption * O.voigt(padded, z, N, num_lines)
    idx = np.nonzero(win)[0]
    w0, w1 = words(seed, g, STREAM_PIXEL, idx)
    e1, e2 = normals(w0, w1)
    out_flux = y_in.copy() if inject else np.full(L, np.nan)
    if inject:
        ex = 1.0 - absorption * absorption
        with np.errstate(invalid="ignore"):
            noise = np.where(ex > 0.0, np.sqrt(np.where(ex > 0.0, ex, 0.0) * v[win]) * e2, 0.0)
        out_flux[win] = absorption * y_in[win] + noise
    else:
        k = model["M"].shape[1]
        lw0, lw1 = words(seed, g, STREAM_LATENT, np.arange(k // 2))
        xa, xb = normals(lw0, lw1)
        xi = np.stack([xa, xb], axis=1).ravel()
        _, _, mu_t, M_t, om2_t = R.window_model(model, w_win, rest[win], z_qso, kind == 1)
        out_flux[win] = absorption * (mu_t + M_t @ xi + np.sqrt(om2_t) * e1) + np.sqrt(v[win]) * e2
    out_abs = np.full(L, np.nan)
    out_abs[win] = absorption
    return dict(flux=out_flux, absorption=out_abs), truth, edge


def draw_spectra(model, samples, prior, spectra, seed, first_quasar=0, kind=0, max_dlas=4, inject=False,
                 absorber_z=None, absorber_nhi=None, num_lines=O.num_lines_default, L_max=None, Z_lls=None, Z_dla=None):
    """Every quasar of ragged ``spectra``: ``flux``, ``absorption`` [Q, L_max] (draw: 0 past each length; inject: the
    input flux there), ``truth_model`` [Q], ``truth_inds``, ``truth_z``, ``truth_log_nhi`` [Q, TW] and ``edge`` [Q],
    each model choice's distance to the nearest cumulative edge."""
    Q = len(spectra["z_qsos"])
    lengths = [len(w) for w in spectra["all_wavelengths"]]
    L_max = max(max(lengths) if Q else 1, 1) if L_max is None else L_max
    TW = max_dlas if kind == 1 else 1
    from_prior = absorber_z is None
    res = dict(flux=np.zeros((Q, L_max)), absorption=np.full((Q, L_max), np.nan),
               truth_model=np.zeros(Q, np.int32), truth_inds=np.full((Q, TW), -1, np.int64),
               truth_z=np.full((Q, TW), np.nan), truth_log_nhi=np.full((Q, TW), np.nan), edge=np.full(Q, np.inf))
    for q in range(Q):
        az = an = ()
        if not from_prior:
            az = np.asarray(absorber_z, dtype=np.float64).reshape(Q, -1)[q]
            an = np.asarray(absorber_nhi, dtype=np.float64).reshape(Q, -1)[q]
        row, truth, edge = draw_one(model, samples, prior, spectra["all_wavelengths"][q], spectra["all_flux"][q],
                                    spectra["all_noise_variance"][q], spectra["all_pixel_mask"][q],
                                    float(spectra["z_qsos"][q]), seed, first_quasar + q, kind, max_dlas, inject, az,
                                    an, from_prior, num_lines, Z_lls, Z_dla)
        n = lengths[q]
        if row is None:                       # no used pixel, or no draw: the whole padded row is NaN
            res["flux"][q] = np.nan
        else:
            res["flux"][q, :n] = row["flux"]
            res["absorption"][q, :n] = row["absorption"]
        res["truth_model"][q] = truth["code"]
        res["truth_inds"][q], res["truth_z"][q], res["truth_log_nhi"][q] = truth["inds"], truth["z"], truth["log_nhi"]
        res["edge"][q] = edge
    return res
