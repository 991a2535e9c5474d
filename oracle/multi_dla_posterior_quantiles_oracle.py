"""NumPy restatement of the credible intervals of every absorber of the multi-DLA model
(``gpdla_multi_dla_posterior_quantiles``).  Test infrastructure only: a literal per-quasar loop over levels and ranks
that ranks every sample's absorbers (``dla_posteriors_oracle.ranked_slots``), then sorts each rank's values and takes
their cumulative weight (``lower_quantile``); it shares none of the kernel's sample permutations or histograms.

Restatement decisions, beyond those of ``dla_posteriors_oracle``:

- per level j and rank r < j, the rank-r values of every sample carry the level's weights w_j; the quantile at p is
  ``lower_quantile`` of them, and ``mass_above_threshold = sum_{log N_r(i) >= t} w_ji / sum w_j``;
- a level with no weight or a partner outside [0, S) is NaN, the other levels are not; ``max_z <= min_z`` makes the
  whole record NaN;
- the kernel accumulates fixed-point weights floor(w 2^F), F = 63 - ceil(log2 S), which move each cumulative fraction by
  at most S 2^-F: its quantiles are held to ``acceptable_quantiles(..., tol=quantile_tolerance(S))``.
"""
from __future__ import annotations

import numpy as np

from oracle.dla_posteriors_oracle import lower_quantile, ranked_slots, weights


def quantile_bits(S):
    """F = 63 - ceil(log2 S): the fixed-point bits of the kernel's weights."""
    return 63 - (int(S) - 1).bit_length()


def quantile_tolerance(S):
    """S 2^-F + 1e-12: how far the kernel's fixed-point cumulative fractions may lie from the float ones (the largest
    weight is 1, so the total weight is at least 1)."""
    return S * 2.0 ** -quantile_bits(S) + 1e-12


def width(J, P):
    return J * (J + 1) // 2 * (1 + 2 * P)


def multi_quasar_posterior_quantiles(ll, part, min_z, max_z, offset, log_nhi, quantiles, threshold=20.3):
    """One quasar of the multi-DLA model, ll [J, S], part [J-1, S]: per level j and rank r < j,
    (mass_above_threshold, z quantiles [P], log-N quantiles [P])."""
    ll = np.asarray(ll, dtype=np.float64)
    J, S = ll.shape
    P = len(quantiles)
    out = []
    for j in range(1, J + 1):
        block = np.full((j, 1 + 2 * P), np.nan)
        w = weights(ll[j - 1])
        rows = np.asarray(part[:j - 1])
        if w is not None and max_z > min_z and not np.any((rows < 0) | (rows >= S)):
            z, n = ranked_slots(part, j, min_z, max_z, offset, log_nhi)
            tot = np.sum(w)
            for r in range(j):
                block[r, 0] = np.sum(w[n[r] >= threshold]) / tot
                for k, p in enumerate(quantiles):
                    block[r, 1 + k] = lower_quantile(z[r], w, p)
                    block[r, 1 + P + k] = lower_quantile(n[r], w, p)
        out.append(block.ravel())
    return np.concatenate(out)


def multi_dla_posterior_quantiles(ll, base_sample_inds, min_z_dlas, max_z_dlas, offset_samples, log_nhi_samples,
                                  quantiles, threshold=20.3):
    """ll [Q, J, S], base_sample_inds [Q, J-1, S] (None when J == 1) -> [Q, J (J + 1) / 2 (1 + 2 P)]."""
    ll = np.asarray(ll, dtype=np.float64)
    Q, J, S = ll.shape
    part = np.zeros((Q, 0, S), dtype=np.int64) if base_sample_inds is None else np.asarray(base_sample_inds)
    return np.stack([multi_quasar_posterior_quantiles(ll[q], part[q], min_z_dlas[q], max_z_dlas[q], offset_samples,
                                                      log_nhi_samples, quantiles, threshold)
                     for q in range(Q)]).reshape(Q, width(J, len(quantiles)))
