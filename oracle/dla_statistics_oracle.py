"""NumPy restatement of the population statistics of the single-DLA catalogue: the additive sums behind the column
density distribution f(N_HI, X), the line density dN/dX and Omega_DLA (CDDF_analysis/calc_cddf.py; Bird, Garnett & Ho
2017), and the host finish.  Test infrastructure only; per-quasar loops and ``searchsorted`` binning.

``calc_cddf.py`` is not in this image, so this restates the statistic from its definition; parity with it is
**unpinned**.  Restatement decisions (each one a parameter or a line below):

- the sample posterior of quasar i is ``w_ij = exp(ll_ij - m_i) / sum_j exp(ll_ij - m_i)``, ``m_i = max_j ll_ij``: the
  samples are prior draws, so this is the posterior over samples given a DLA; each sample enters with weight
  ``p_dla_i w_ij``;
- a quasar contributes (counts, variances, path and ``num_quasars``) iff ``select[i]``, ``isfinite(p_dla)``,
  ``max_z_dla > min_z_dla`` and the row's log-sum-exp is finite; otherwise it contributes nothing;
- ``z_ij = min_z + (max_z - min_z) offset_j`` with each operation rounded (as ``map_z_dlas``); ``log N_j`` and ``N_j``
  are the stored samples;
- bins are half-open ``[lo, hi)``; a sample is a DLA where ``log N_j >= dla_log_nhi_min`` (default 20.3);
- variances are the exact Poisson-binomial ones, ``sum q (1 - q)``, and ``sum (e2 - e^2)`` for the N_HI sum;
- absorption distance of flat LambdaCDM without radiation, ``X(z) = 2 / (3 Omega_m) sqrt(Omega_m (1+z)^3 + 1 -
  Omega_m)``, clipped to ``[min_z, max_z]`` of each quasar;
- ``Omega_DLA = 8 pi G m_H / (3 c H0) sum N / path`` with the hydrogen-atom mass m_H and no helium correction.
"""
from __future__ import annotations

import math

import numpy as np

G = 6.67430e-8                       # cm^3 g^-1 s^-2, CODATA 2018
C = 2.99792458e10                    # cm / s
M_H = 1.6735575e-24                  # g
MPC = 3.0856775814913673e24          # cm


def absorption_distance(z, omega_m):
    """X(z) with the operations in the kernel's order: coef * sqrt(om * ((a * a) * a) + ol), a = 1 + z."""
    a = 1.0 + np.asarray(z, dtype=np.float64)
    return (2.0 / (3.0 * omega_m)) * np.sqrt(omega_m * ((a * a) * a) + (1.0 - omega_m))


def path_length(min_z, max_z, lo, hi, omega_m):
    """dX of one quasar in the z bin [lo, hi): max(0, X(min(hi, max_z)) - X(max(lo, min_z)))."""
    return max(0.0, float(absorption_distance(min(hi, max_z), omega_m) - absorption_distance(max(lo, min_z), omega_m)))


def contributes(ll_row, p_dla, min_z, max_z, selected=True) -> bool:
    if not selected or not np.isfinite(p_dla) or not (max_z > min_z):
        return False
    if np.any(np.isnan(ll_row)):
        return False
    m = np.max(ll_row)
    return bool(np.isfinite(m))


def quasar_cells(ll_row, p_dla, min_z, max_z, offset, log_nhi, nhi, z_edges, log_nhi_edges,
                 dla_log_nhi_min=20.3):
    """Per-quasar cell values: q [n_z, n_nhi], d, e, e2 [n_z] (steps 2-4)."""
    z_edges, log_nhi_edges = np.asarray(z_edges, float), np.asarray(log_nhi_edges, float)
    n_z, n_nhi = z_edges.size - 1, log_nhi_edges.size - 1
    m = np.max(ll_row)
    w = np.exp(ll_row - m)
    w = w / np.sum(w)
    z = min_z + (max_z - min_z) * np.asarray(offset, float)        # numpy rounds each operation
    b = np.searchsorted(z_edges, z, side="right") - 1
    c = np.searchsorted(log_nhi_edges, log_nhi, side="right") - 1
    inz = (b >= 0) & (b < n_z)
    innhi = (c >= 0) & (c < n_nhi)
    dla = np.asarray(log_nhi) >= dla_log_nhi_min
    q = np.zeros((n_z, n_nhi))
    d, e, e2 = np.zeros(n_z), np.zeros(n_z), np.zeros(n_z)
    for j in range(w.size):
        if not inz[j]:
            continue
        if innhi[j]:
            q[b[j], c[j]] += w[j]
        if dla[j]:
            d[b[j]] += w[j]
            e[b[j]] += w[j] * nhi[j]
            e2[b[j]] += w[j] * nhi[j] * nhi[j]
    return p_dla * q, p_dla * d, p_dla * e, p_dla * e2


def dla_statistics_sums(ll, p_dlas, min_z_dlas, max_z_dlas, offset_samples, log_nhi_samples, nhi_samples, z_edges,
                        log_nhi_edges, select=None, dla_log_nhi_min=20.3, omega_m=0.3, sums=None):
    """The sums vector in the library's layout (steps 1-6), quasar by quasar."""
    z_edges, log_nhi_edges = np.asarray(z_edges, float), np.asarray(log_nhi_edges, float)
    n_z, n_nhi = z_edges.size - 1, log_nhi_edges.size - 1
    ll = np.asarray(ll, float)
    Q = ll.shape[0]
    counts, counts_var = np.zeros((n_z, n_nhi)), np.zeros((n_z, n_nhi))
    dla, dla_var, nh, nh_var, path = (np.zeros(n_z) for _ in range(5))
    nq = 0
    for i in range(Q):
        sel = True if select is None else bool(select[i])
        if not contributes(ll[i], p_dlas[i], min_z_dlas[i], max_z_dlas[i], sel):
            continue
        q, d, e, e2 = quasar_cells(ll[i], p_dlas[i], min_z_dlas[i], max_z_dlas[i], offset_samples, log_nhi_samples,
                                   nhi_samples, z_edges, log_nhi_edges, dla_log_nhi_min)
        counts += q
        counts_var += q * (1.0 - q)
        dla += d
        dla_var += d * (1.0 - d)
        nh += e
        nh_var += e2 - e * e
        for b in range(n_z):
            path[b] += path_length(min_z_dlas[i], max_z_dlas[i], z_edges[b], z_edges[b + 1], omega_m)
        nq += 1
    out = np.concatenate([counts.ravel(), counts_var.ravel(), dla, dla_var, nh, nh_var, path, [float(nq)]])
    return out if sums is None else np.asarray(sums, float) + out


def omega_coefficient(hubble_h=0.7):
    H0 = 100.0 * hubble_h * 1e5 / MPC
    return 8.0 * math.pi * G * M_H / (3.0 * C * H0)


def finish(sums, z_edges, log_nhi_edges, hubble_h=0.7):
    """Step 7: f(N), dN/dX, Omega_DLA and their sigmas from the sums."""
    z_edges, log_nhi_edges = np.asarray(z_edges, float), np.asarray(log_nhi_edges, float)
    n_z, n_nhi = z_edges.size - 1, log_nhi_edges.size - 1
    a = n_z * n_nhi
    counts, counts_var = sums[:a].reshape(n_z, n_nhi), sums[a:2 * a].reshape(n_z, n_nhi)
    dla, dla_var, nh, nh_var, path = (sums[2 * a + k * n_z:2 * a + (k + 1) * n_z] for k in range(5))
    dn = 10.0 ** log_nhi_edges[1:] - 10.0 ** log_nhi_edges[:-1]
    k = omega_coefficient(hubble_h)
    out = dict(cddf=np.zeros((n_z, n_nhi)), cddf_sigma=np.zeros((n_z, n_nhi)), dndx=np.zeros(n_z),
               dndx_sigma=np.zeros(n_z), omega_dla=np.zeros(n_z), omega_dla_sigma=np.zeros(n_z))
    for b in range(n_z):
        for c in range(n_nhi):
            out["cddf"][b, c] = counts[b, c] / (dn[c] * path[b])
            out["cddf_sigma"][b, c] = math.sqrt(counts_var[b, c]) / (dn[c] * path[b])
        out["dndx"][b] = dla[b] / path[b]
        out["dndx_sigma"][b] = math.sqrt(dla_var[b]) / path[b]
        out["omega_dla"][b] = k * nh[b] / path[b]
        out["omega_dla_sigma"][b] = k * math.sqrt(nh_var[b]) / path[b]
    return out
