"""NumPy restatement of the per-quasar absorber posterior summaries (``gpdla_dla_posteriors`` and
``gpdla_multi_dla_posteriors``).  Test infrastructure only: a literal per-quasar loop that sorts every row by value
(``np.argsort(kind="stable")``), takes the cumulative sum, and for the multi-DLA model enumerates every sample's slots;
it shares none of the kernels' permutations, chunked scans or sorting network.

Restatement decisions:

- the sample posterior of a quasar is ``w_i = exp(ll_i - m)``, ``m`` the maximum over the entries ``> -inf``; NaN and
  ``-inf`` entries weigh 0.  The samples are prior draws, so this is the DLA-model posterior over the sample set
  (``process_qsos.m:203-210``).  A quasar with no such entry, a non-finite ``m``, or ``max_z <= min_z`` gets NaN;
- ``z_i = min_z + (max_z - min_z) * offset_i`` with each operation rounded (as ``map_z_dlas``);
- ``ess = (sum w)^2 / sum w^2`` (Kish); moments are two-pass: the weighted means, then the weighted central sums,
  divided by ``sum w`` (population moments of the posterior, not sample estimates);
- the quantile at ``p`` is the value of the first sample, in stable value order, whose cumulative weight
  ``cumsum(w)`` reaches ``p * cumsum(w)[-1]``;
- ``mass_above_threshold = sum_{log N_i >= t} w_i / sum w``;
- multi-DLA: sample i of level j places j absorbers, at ``i, base_sample_inds[0, i], ..., base_sample_inds[j-2, i]``
  (``multi_dla_statistics_oracle``); per sample they are ranked by ascending z, ties by log N, then slot; a level with
  no weight or a partner outside [0, S) is NaN, the other levels are not.
"""
from __future__ import annotations

import numpy as np

FIELDS = ["ess", "z_mean", "z_sd", "log_nhi_mean", "log_nhi_sd", "z_log_nhi_cov", "mass_above_threshold"]


def weights(ll_row):
    """w = exp(ll - max) over the entries > -inf, 0 elsewhere; None when no entry carries finite weight."""
    ll_row = np.asarray(ll_row, dtype=np.float64)
    ok = ll_row > -np.inf
    if not np.any(ok):
        return None
    m = np.max(ll_row[ok])
    if not np.isfinite(m):
        return None
    return np.where(ok, np.exp(np.where(ok, ll_row, m) - m), 0.0)


def sample_z(min_z, max_z, offset):
    return min_z + (max_z - min_z) * np.asarray(offset, dtype=np.float64)   # numpy rounds each operation


def moments(w, x):
    """(mean, standard deviation) of x under weights w, two-pass."""
    tot = np.sum(w)
    mean = np.sum(w * x) / tot
    return mean, np.sqrt(np.sum(w * (x - mean) ** 2) / tot)


def lower_quantile(values, w, p):
    """The value of the first sample, in stable value order, whose cumulative weight reaches p * total."""
    order = np.argsort(values, kind="stable")
    c = np.cumsum(w[order])
    return values[order][int(np.searchsorted(c, p * c[-1], side="left"))]


def acceptable_quantiles(values, w, p, tol=1e-12):
    """The values a kernel may report at p when its cumulative sums differ from np.cumsum by rounding: every sample
    j with cumsum[j] >= target - tol * total and cumsum[j-1] < target + tol * total.  Returns (values, ambiguous)."""
    order = np.argsort(values, kind="stable")
    c = np.cumsum(w[order])
    t, slack = p * c[-1], tol * c[-1]
    prev = np.concatenate([[-np.inf], c[:-1]])
    ok = (c >= t - slack) & (prev < t + slack)
    vals = np.unique(values[order][ok])
    return vals, vals.size > 1


def quasar_posterior(ll_row, min_z, max_z, offset, log_nhi, quantiles, threshold=20.3):
    """One quasar's record: FIELDS, then the z quantiles, then the log-N quantiles."""
    P = len(quantiles)
    rec = np.full(len(FIELDS) + 2 * P, np.nan)
    w = weights(ll_row)
    if w is None or not (max_z > min_z):
        return rec
    z, n = sample_z(min_z, max_z, offset), np.asarray(log_nhi, dtype=np.float64)
    tot = np.sum(w)
    zm, zsd = moments(w, z)
    nm, nsd = moments(w, n)
    rec[0] = tot * tot / np.sum(w * w)
    rec[1:5] = zm, zsd, nm, nsd
    rec[5] = np.sum(w * (z - zm) * (n - nm)) / tot
    rec[6] = np.sum(w[n >= threshold]) / tot
    for k, p in enumerate(quantiles):
        rec[7 + k] = lower_quantile(z, w, p)
        rec[7 + P + k] = lower_quantile(n, w, p)
    return rec


def dla_posteriors(ll, min_z_dlas, max_z_dlas, offset_samples, log_nhi_samples, quantiles, threshold=20.3):
    """[Q, 7 + 2 P], quasar by quasar."""
    ll = np.asarray(ll, dtype=np.float64)
    return np.stack([quasar_posterior(ll[q], min_z_dlas[q], max_z_dlas[q], offset_samples, log_nhi_samples, quantiles,
                                      threshold) for q in range(ll.shape[0])]).reshape(ll.shape[0], -1)


def ranked_slots(part, j, min_z, max_z, offset, log_nhi):
    """(z, log N) [j, S] of the j absorbers of every sample of level j, ranked by ascending z, then log N, then slot."""
    S = np.asarray(offset).size
    slots = np.concatenate([np.arange(S)[None, :], np.asarray(part[:j - 1], dtype=np.int64)])
    z = sample_z(min_z, max_z, offset)[slots]
    n = np.asarray(log_nhi, dtype=np.float64)[slots]
    slot_id = np.broadcast_to(np.arange(j)[:, None], slots.shape)
    order = np.lexsort((slot_id, n, z), axis=0)                 # the last key is the primary one
    return np.take_along_axis(z, order, axis=0), np.take_along_axis(n, order, axis=0)


def multi_quasar_posterior(ll, part, min_z, max_z, offset, log_nhi):
    """One quasar of the multi-DLA model, ll [J, S], part [J-1, S]: per level j, ess_j then (z_mean, z_sd,
    log_nhi_mean, log_nhi_sd) of ranks 0..j-1."""
    J, S = ll.shape
    out = []
    for j in range(1, J + 1):
        block = np.full(1 + 4 * j, np.nan)
        w = weights(ll[j - 1])
        rows = np.asarray(part[:j - 1])
        if w is not None and max_z > min_z and not np.any((rows < 0) | (rows >= S)):
            z, n = ranked_slots(part, j, min_z, max_z, offset, log_nhi)
            block[0] = np.sum(w) ** 2 / np.sum(w * w)
            for r in range(j):
                block[1 + 4 * r:5 + 4 * r] = moments(w, z[r]) + moments(w, n[r])
        out.append(block)
    return np.concatenate(out)


def multi_dla_posteriors(ll, base_sample_inds, min_z_dlas, max_z_dlas, offset_samples, log_nhi_samples):
    """ll [Q, J, S], base_sample_inds [Q, J-1, S] (None when J == 1) -> [Q, J + 2 J (J + 1)]."""
    ll = np.asarray(ll, dtype=np.float64)
    Q, J, S = ll.shape
    part = np.zeros((Q, 0, S), dtype=np.int64) if base_sample_inds is None else np.asarray(base_sample_inds)
    return np.stack([multi_quasar_posterior(ll[q], part[q], min_z_dlas[q], max_z_dlas[q], offset_samples,
                                            log_nhi_samples) for q in range(Q)]).reshape(Q, -1)
