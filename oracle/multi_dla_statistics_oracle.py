"""NumPy restatement of the population statistics of the multi-DLA catalogue (Ho et al. 2021): the additive sums
behind f(N_HI, X), dN/dX and Omega_DLA when a quasar may hold up to J DLAs.  Test infrastructure only; it enumerates
every sample's absorbers per level and does not use the kernel's slot / pair decomposition, so it checks it.

Inputs are one ``process_multi`` call's outputs in the C layout: ``ll`` [Q, J, S] (sample_log_likelihoods_dla),
``base_sample_inds`` [Q, J-1, S] (0-based), ``model_posteriors`` [Q, 2 + J] (no DLA, sub-DLA, 1..J DLAs).

Parity with ``calc_cddf.py`` is **unpinned**.  Restatement decisions:

- the quasar's model is a mixture: model M with probability ``p_M = model_posteriors[q, M]``; under the j-DLA model,
  sample i with probability ``w_ji = exp(ll_ji - m_j) / sum_i' exp(ll_ji' - m_j)``, ``m_j`` the max over the non-NaN
  entries.  NaN entries (the z-separation filter's) weigh 0, as the reference's ``nanmax`` / ``nanmean`` ignore them;
  the Occam term ``-log S`` cancels;
- sample i of level j places j absorbers, at samples ``i, base_sample_inds[0, i], ..., base_sample_inds[j-2, i]``; the
  no-DLA and **sub-DLA models place none**;
- a quasar contributes (counts, variances, path and ``num_quasars``) iff ``select[q]``, every entry of its
  ``model_posteriors`` row is finite, ``max_z > min_z``, and every level with ``p_j > 0`` has a finite ``m_j`` and
  partner indices in [0, S); otherwise it contributes nothing.  Levels with ``p_j == 0`` are skipped;
- per quasar the counts X (absorbers in a (z, log N) cell), D (absorbers in a z bin with log N >= dla_log_nhi_min)
  and E (their N_HI sum) enter with their **exact mixture mean and variance**, ``Var = E[X^2] - E[X]^2``, not a
  per-absorber Poisson-binomial one; with J = 1 this is the single-DLA statistic;
- the single-DLA decisions carry over (``dla_statistics_oracle``): z of an absorber rounded as ``map_z_dlas``,
  half-open bins, flat LambdaCDM path, m_H with no helium.
"""
from __future__ import annotations

import numpy as np

from .dla_statistics_oracle import path_length


def contributes(ll, base_sample_inds, model_posteriors, min_z, max_z, selected=True) -> bool:
    """ll [J, S], base_sample_inds [J-1, S], model_posteriors [2 + J] of one quasar."""
    post = np.asarray(model_posteriors, float)
    if not selected or not np.all(np.isfinite(post)) or not (max_z > min_z):
        return False
    J, S = ll.shape
    for j in range(1, J + 1):
        if not post[1 + j] > 0:
            continue
        row = ll[j - 1]
        if np.all(np.isnan(row)) or not np.isfinite(np.nanmax(row)):
            return False
        part = np.asarray(base_sample_inds[:j - 1])
        if np.any((part < 0) | (part >= S)):
            return False
    return True


def quasar_moments(ll, base_sample_inds, model_posteriors, min_z, max_z, offset, log_nhi, nhi, z_edges, log_nhi_edges,
                   dla_log_nhi_min=20.3):
    """E[X], E[X^2] per (z, log N) cell [n_z, n_nhi]; E[D], E[D^2], E[E], E[E^2] per z bin [n_z]."""
    z_edges, log_nhi_edges = np.asarray(z_edges, float), np.asarray(log_nhi_edges, float)
    n_z, n_nhi = z_edges.size - 1, log_nhi_edges.size - 1
    ncell = n_z * n_nhi
    J, S = ll.shape
    z = min_z + (max_z - min_z) * np.asarray(offset, float)        # numpy rounds each operation
    b = np.searchsorted(z_edges, z, side="right") - 1
    c = np.searchsorted(log_nhi_edges, log_nhi, side="right") - 1
    inz = (b >= 0) & (b < n_z)
    cell = np.where(inz & (c >= 0) & (c < n_nhi), b * n_nhi + c, -1)   # cell of an absorber at sample s
    zbin = np.where(inz & (np.asarray(log_nhi) >= dla_log_nhi_min), b, -1)
    nhi = np.asarray(nhi, float)
    ex, ex2 = np.zeros(ncell), np.zeros(ncell)
    ed, ed2, ee, ee2 = (np.zeros(n_z) for _ in range(4))
    for j in range(1, J + 1):
        p = float(model_posteriors[1 + j])
        if not p > 0:
            continue
        row = ll[j - 1]
        ok = ~np.isnan(row)
        w = np.where(ok, np.exp(np.where(ok, row, 0.0) - np.nanmax(row)), 0.0)
        w = w / np.sum(w)
        # the j absorbers of every sample: slots[t, i] is the sample at which absorber t of sample i sits
        slots = np.concatenate([np.arange(S)[None, :], np.asarray(base_sample_inds[:j - 1], dtype=np.int64)])
        owner = np.broadcast_to(np.arange(S), slots.shape)
        # x = the number of sample i's absorbers in each cell, for every (sample, cell) pair that has one
        ck = cell[slots]
        v = ck >= 0
        keys, x = np.unique(owner[v] * ncell + ck[v], return_counts=True)
        i_of, c_of = np.divmod(keys, ncell)
        ex += p * np.bincount(c_of, weights=w[i_of] * x, minlength=ncell)
        ex2 += p * np.bincount(c_of, weights=w[i_of] * x * x, minlength=ncell)
        # D and E per (sample, z bin)
        zk = zbin[slots]
        v = zk >= 0
        keys, inv = np.unique(owner[v] * n_z + zk[v], return_inverse=True)
        d = np.bincount(inv).astype(float)
        e = np.bincount(inv, weights=nhi[slots[v]])
        i_of, b_of = np.divmod(keys, n_z)
        ed += p * np.bincount(b_of, weights=w[i_of] * d, minlength=n_z)
        ed2 += p * np.bincount(b_of, weights=w[i_of] * d * d, minlength=n_z)
        ee += p * np.bincount(b_of, weights=w[i_of] * e, minlength=n_z)
        ee2 += p * np.bincount(b_of, weights=w[i_of] * e * e, minlength=n_z)
    return ex.reshape(n_z, n_nhi), ex2.reshape(n_z, n_nhi), ed, ed2, ee, ee2


def multi_dla_statistics_sums(ll, base_sample_inds, model_posteriors, min_z_dlas, max_z_dlas, offset_samples,
                              log_nhi_samples, nhi_samples, z_edges, log_nhi_edges, select=None, dla_log_nhi_min=20.3,
                              omega_m=0.3, sums=None):
    """The sums vector in the library's layout (``dla_statistics_layout``), quasar by quasar."""
    z_edges, log_nhi_edges = np.asarray(z_edges, float), np.asarray(log_nhi_edges, float)
    n_z, n_nhi = z_edges.size - 1, log_nhi_edges.size - 1
    ll = np.asarray(ll, float)
    Q, J, S = ll.shape
    part = np.zeros((Q, 0, S), dtype=np.int64) if base_sample_inds is None else np.asarray(base_sample_inds)
    counts, counts_var = np.zeros((n_z, n_nhi)), np.zeros((n_z, n_nhi))
    dla, dla_var, nh, nh_var, path = (np.zeros(n_z) for _ in range(5))
    nq = 0
    for q in range(Q):
        sel = True if select is None else bool(select[q])
        if not contributes(ll[q], part[q], model_posteriors[q], min_z_dlas[q], max_z_dlas[q], sel):
            continue
        ex, ex2, ed, ed2, ee, ee2 = quasar_moments(ll[q], part[q], model_posteriors[q], min_z_dlas[q], max_z_dlas[q],
                                                   offset_samples, log_nhi_samples, nhi_samples, z_edges,
                                                   log_nhi_edges, dla_log_nhi_min)
        counts += ex
        counts_var += ex2 - ex * ex
        dla += ed
        dla_var += ed2 - ed * ed
        nh += ee
        nh_var += ee2 - ee * ee
        for b in range(n_z):
            path[b] += path_length(min_z_dlas[q], max_z_dlas[q], z_edges[b], z_edges[b + 1], omega_m)
        nq += 1
    out = np.concatenate([counts.ravel(), counts_var.ravel(), dla, dla_var, nh, nh_var, path, [float(nq)]])
    return out if sums is None else np.asarray(sums, float) + out
