"""Quasar sharding across the GPUs of one box.

The reference parallelises by hand: ``test_ind`` selects a slice of quasars per SLURM job and
``CDDF_analysis/sbatch_reunion.py:13-63`` concatenates the per-job files.  Here the same split
is a contiguous partition of the catalogue balanced by per-quasar cost (number of pixels in the
modelled window x samples); every rank (one process per GPU) runs the hot path on its block with
no data-path collective, and ONE ``all_gather`` of fixed-width per-quasar records (NCCL over
NVLink on GPUs, gloo in CPU tests) reassembles the catalogue.  ``sample_log_likelihoods_dla``
(80 KB/quasar) stays sharded; ``dla_statistics_sharded`` (and ``multi_dla_statistics_sharded`` for the multi-DLA
model) reduces it to the population-statistics sums on the rank that produced it and gathers only those (a few KB);
``dla_posteriors_sharded`` (and ``multi_dla_posteriors_sharded``) reduces it to fixed-width posterior summaries per
quasar and gathers those.
"""
from __future__ import annotations

from typing import Callable, Dict, List, Sequence, Tuple

import numpy as np

RECORD_F64 = ["min_z_dlas", "max_z_dlas", "log_priors_no_dla", "log_priors_dla", "log_likelihoods_no_dla",
              "log_likelihoods_dla", "log_posteriors_no_dla", "log_posteriors_dla", "p_no_dlas", "p_dlas",
              "map_z_dlas", "map_log_nhis"]
RECORD_WIDTH = len(RECORD_F64) + 3   # + model_posteriors (2) + map_inds (1, int64 bit pattern)


def partition_by_cost(costs: Sequence[float], world_size: int) -> List[Tuple[int, int]]:
    """Contiguous blocks ``[start, end)`` whose summed cost is as equal as prefix sums allow."""
    costs = np.asarray(costs, dtype=np.float64)
    Q = costs.size
    if world_size < 1:
        raise ValueError("world_size must be >= 1")
    csum = np.concatenate([[0.0], np.cumsum(costs)])
    total = csum[-1]
    bounds = [0]
    for r in range(1, world_size):
        target = total * r / world_size
        j = int(np.searchsorted(csum, target, side="left"))
        if j > 0 and abs(csum[j - 1] - target) <= abs(csum[min(j, Q)] - target):
            j -= 1
        bounds.append(min(max(j, bounds[-1]), Q))
    bounds.append(Q)
    return [(bounds[r], bounds[r + 1]) for r in range(world_size)]


def quasar_costs(spectra: Dict, min_lambda: float = 911.75, max_lambda: float = 1215.75) -> np.ndarray:
    """Pixels inside the modelled rest-frame window per quasar (cost of one quasar ~ n_u x samples)."""
    if "lengths" in spectra:
        W, L, z = spectra["wavelengths"], spectra["lengths"], spectra["z_qsos"]
        rest = W / (1.0 + np.asarray(z)[:, None])
        valid = np.arange(W.shape[1])[None, :] < np.asarray(L)[:, None]
        return np.count_nonzero(valid & (rest >= min_lambda) & (rest <= max_lambda), axis=1).astype(np.float64)
    return np.array([np.count_nonzero((w / (1 + z) >= min_lambda) & (w / (1 + z) <= max_lambda))
                     for w, z in zip(spectra["all_wavelengths"], spectra["z_qsos"])], dtype=np.float64)


def slice_spectra(spectra: Dict, start: int, end: int) -> Dict:
    if "lengths" in spectra:
        return {k: v[start:end] for k, v in spectra.items()}
    return {k: (v[start:end] if k in ("all_wavelengths", "all_flux", "all_noise_variance", "all_pixel_mask", "z_qsos")
                else v) for k, v in spectra.items()}


def pack_records(res: Dict[str, np.ndarray]) -> np.ndarray:
    """Per-quasar results -> ``[Q_local x RECORD_WIDTH]`` float64 (map_inds carried as its bit pattern)."""
    Q = len(res["p_dlas"])
    rec = np.empty((Q, RECORD_WIDTH), dtype=np.float64)
    for i, n in enumerate(RECORD_F64):
        rec[:, i] = res[n]
    rec[:, len(RECORD_F64):len(RECORD_F64) + 2] = res["model_posteriors"]
    rec[:, -1] = np.asarray(res["map_inds"], dtype=np.int64).view(np.float64)
    return rec


def unpack_records(rec: np.ndarray) -> Dict[str, np.ndarray]:
    out = {n: rec[:, i].copy() for i, n in enumerate(RECORD_F64)}
    out["model_posteriors"] = rec[:, len(RECORD_F64):len(RECORD_F64) + 2].copy()
    out["map_inds"] = rec[:, -1].copy().view(np.int64)
    return out


def gather_records(local: np.ndarray, blocks: List[Tuple[int, int]], device=None, width: int = RECORD_WIDTH) -> np.ndarray:
    """One all_gather of the padded record blocks; returns the catalogue-ordered ``[Q x width]``."""
    import torch
    import torch.distributed as dist
    world = dist.get_world_size()
    qmax = max(e - s for s, e in blocks)
    buf = torch.zeros((max(qmax, 1), width), dtype=torch.float64, device=device)
    if local.shape[0]:
        buf[:local.shape[0]] = torch.from_numpy(local).to(buf.device)
    out = torch.empty((world * buf.shape[0], width), dtype=torch.float64, device=device)
    dist.all_gather_into_tensor(out, buf)
    out = out.cpu().numpy().reshape(world, buf.shape[0], width)
    return np.concatenate([out[r, :e - s] for r, (s, e) in enumerate(blocks)], axis=0)


def process_qsos_sharded(model: Dict, samples: Dict, spectra: Dict, prior: Dict, params=None,
                         compute: Callable[[Dict], Dict[str, np.ndarray]] = None, device=None) -> Dict:
    """Every rank calls this with the FULL catalogue description; rank r processes block r and all
    ranks return the gathered per-quasar results.  ``compute`` defaults to the CUDA path on
    ``cuda:LOCAL_RANK``; tests inject a CPU stand-in to exercise the partition/gather logic."""
    import torch.distributed as dist
    rank, world = dist.get_rank(), dist.get_world_size()
    blocks = partition_by_cost(quasar_costs(spectra), world)
    s, e = blocks[rank]
    mine = slice_spectra(spectra, s, e)
    if compute is None:
        import os
        from .api import DLAProcessor
        from .params import DEFAULT
        proc = DLAProcessor(model, samples, prior, params or DEFAULT, device=int(os.environ.get("LOCAL_RANK", 0)))
        compute = lambda sp: proc.process(sp, return_sample_log_likelihoods=False)
    if e > s:
        rec = pack_records(compute(mine))
    else:
        rec = np.zeros((0, RECORD_WIDTH))
    full = gather_records(rec, blocks, device=device)
    out = unpack_records(full)
    out["blocks"] = blocks
    return out


def gather_sums(local: np.ndarray, device=None) -> np.ndarray:
    """One all_gather of every rank's fixed-width sums vector, added in rank order: every rank gets the same bits."""
    import torch
    import torch.distributed as dist
    world = dist.get_world_size()
    buf = torch.from_numpy(np.ascontiguousarray(local, dtype=np.float64)).to(device or "cpu")
    out = torch.empty(world * buf.numel(), dtype=torch.float64, device=buf.device)
    dist.all_gather_into_tensor(out, buf)
    parts = out.cpu().numpy().reshape(world, buf.numel())
    total = parts[0].copy()
    for r in range(1, world):
        total += parts[r]
    return total


def dla_statistics_sharded(model: Dict, samples: Dict, spectra: Dict, prior: Dict, z_edges, log_nhi_edges,
                           select=None, params=None, batch_quasars: int = 4096, dla_log_nhi_min: float = None,
                           omega_m: float = None, hubble_h: float = None,
                           compute: Callable[[Dict, np.ndarray, np.ndarray], np.ndarray] = None, device=None) -> Dict:
    """Population statistics (``api.finish_dla_statistics``) of the whole catalogue on every rank.  Every rank calls
    this with the FULL catalogue description (and ``select`` [Q], optional); rank r runs its cost-balanced block through
    ``process_device`` in batches of ``batch_quasars`` and accumulates the sums on its GPU with ``statistics_device``;
    one ``all_gather`` of the fixed-width vector follows, added in rank order.  The bits depend on the batch split and
    the world size (they set the summation order); repeated runs with the same ones are identical.  ``compute(spectra,
    select, sums) -> sums`` replaces the CUDA path of one rank (tests inject a CPU stand-in); the CUDA path keeps the
    sums on the GPU between batches.  Returns the finished
    dict plus ``sums`` and ``blocks``."""
    from . import params as P
    dla_log_nhi_min = P.dla_log_nhi_min if dla_log_nhi_min is None else dla_log_nhi_min
    omega_m = P.omega_m if omega_m is None else omega_m
    if compute is None:
        compute = _device_statistics(model, samples, prior, params, z_edges, log_nhi_edges, dla_log_nhi_min, omega_m)
    return _statistics_sharded(spectra, z_edges, log_nhi_edges, select, batch_quasars, hubble_h, compute, device)


def multi_dla_statistics_sharded(model: Dict, samples: Dict, spectra: Dict, prior: Dict, z_edges, log_nhi_edges,
                                 select=None, params=None, max_dlas: int = 4, batch_quasars: int = 4096,
                                 dla_log_nhi_min: float = None, omega_m: float = None, hubble_h: float = None,
                                 compute: Callable[[Dict, np.ndarray, np.ndarray], np.ndarray] = None,
                                 device=None) -> Dict:
    """``dla_statistics_sharded`` for the multi-DLA model: rank r runs its block through ``process_multi_device`` (up
    to ``max_dlas`` DLAs, sub-DLA model, mean flux; ``samples`` holds the sub-DLA samples) in batches and accumulates
    ``multi_statistics_device`` sums on its GPU; one ``all_gather``, added in rank order.  ``compute`` as there."""
    from . import params as P
    dla_log_nhi_min = P.dla_log_nhi_min if dla_log_nhi_min is None else dla_log_nhi_min
    omega_m = P.omega_m if omega_m is None else omega_m
    if compute is None:
        compute = _device_statistics(model, samples, prior, params, z_edges, log_nhi_edges, dla_log_nhi_min, omega_m,
                                     max_dlas=max_dlas)
    return _statistics_sharded(spectra, z_edges, log_nhi_edges, select, batch_quasars, hubble_h, compute, device)


def _statistics_sharded(spectra, z_edges, log_nhi_edges, select, batch_quasars, hubble_h, compute, device) -> Dict:
    """The cost-balanced block of this rank in batches through ``compute``, one gather of the sums, the finish."""
    import torch.distributed as dist
    from . import params as P
    from .api import dla_statistics_width, finish_dla_statistics
    hubble_h = P.hubble_h if hubble_h is None else hubble_h
    rank, world = dist.get_rank(), dist.get_world_size()
    blocks = partition_by_cost(quasar_costs(spectra), world)
    s, e = blocks[rank]
    Q = len(spectra["z_qsos"])
    sel = np.ones(Q, dtype=bool) if select is None else np.asarray(select, dtype=bool).ravel()
    local = np.zeros(dla_statistics_width(len(z_edges) - 1, len(log_nhi_edges) - 1))
    for b0 in range(s, e, max(int(batch_quasars), 1)):
        b1 = min(e, b0 + max(int(batch_quasars), 1))
        local = compute(slice_spectra(spectra, b0, b1), sel[b0:b1], local)
    if hasattr(local, "cpu"):
        local = local.cpu().numpy()
    total = gather_sums(np.asarray(local, dtype=np.float64), device=device)
    out = finish_dla_statistics(total, z_edges, log_nhi_edges, hubble_h=hubble_h)
    out["sums"] = total
    out["blocks"] = blocks
    return out


def _device_statistics(model, samples, prior, params, z_edges, log_nhi_edges, dla_log_nhi_min, omega_m, max_dlas=0):
    """The CUDA path of one rank: spectra -> process_device -> statistics_device (``max_dlas`` 0), or
    process_multi_device -> multi_statistics_device, into one device sums tensor."""
    import os
    import torch
    from .api import DLAProcessor, pad_spectra
    from .params import DEFAULT
    dev = int(os.environ.get("LOCAL_RANK", 0))
    proc = DLAProcessor(model, samples, prior, params or DEFAULT, device=dev)
    state = {}

    def compute(sp, sel, sums):
        pad = pad_spectra(sp)
        d = torch.device("cuda", dev)
        up = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dtype=dt)).to(d)
        if "sums" not in state:
            state["sums"] = up(sums, np.float64)
        planes = (up(pad["wavelengths"], np.float64), up(pad["flux"], np.float64),
                  up(pad["noise_variance"], np.float64), up(pad["pixel_mask"], np.uint8),
                  up(pad["lengths"], np.int32), up(pad["z_qsos"], np.float64))
        if max_dlas:
            out = proc.process_multi_device(*planes, max_dlas=max_dlas, return_samples=True)
            proc.multi_statistics_device(out, z_edges, log_nhi_edges, select=up(sel, np.uint8), sums=state["sums"],
                                         dla_log_nhi_min=dla_log_nhi_min, omega_m=omega_m)
        else:
            out = proc.process_device(*planes, return_sample_log_likelihoods=True)
            proc.statistics_device(out, z_edges, log_nhi_edges, select=up(sel, np.uint8), sums=state["sums"],
                                   dla_log_nhi_min=dla_log_nhi_min, omega_m=omega_m)
        return state["sums"]
    return compute


def dla_posteriors_sharded(model: Dict, samples: Dict, spectra: Dict, prior: Dict, quantiles=None,
                           log_nhi_threshold: float = None, params=None, batch_quasars: int = 4096,
                           compute: Callable[[Dict], np.ndarray] = None, device=None) -> Dict:
    """Per-quasar posterior summaries (``api.dla_posteriors``) of the whole catalogue on every rank.  Every rank calls
    this with the FULL catalogue description; rank r runs its cost-balanced block through ``process_device`` and
    ``posteriors_device`` in batches of ``batch_quasars``, and one ``all_gather`` of the fixed-width records follows.
    ``compute(spectra) -> records`` replaces the CUDA path of one rank (tests inject a CPU stand-in).  Returns
    ``records`` [Q x (7 + 2 P)] in catalogue order (``api.unpack_dla_posteriors``) and ``blocks``."""
    import torch.distributed as dist
    from . import params as P
    from .api import DEFAULT_QUANTILES, dla_posteriors_width
    quantiles = np.asarray(DEFAULT_QUANTILES if quantiles is None else quantiles, dtype=np.float64).ravel()
    log_nhi_threshold = P.dla_log_nhi_min if log_nhi_threshold is None else log_nhi_threshold
    rank, world = dist.get_rank(), dist.get_world_size()
    blocks = partition_by_cost(quasar_costs(spectra), world)
    s, e = blocks[rank]
    width = dla_posteriors_width(quantiles.size)
    if compute is None and e > s:
        compute = _device_posteriors(model, samples, prior, params, quantiles, log_nhi_threshold)
    step = max(int(batch_quasars), 1)
    parts = [np.asarray(compute(slice_spectra(spectra, b0, min(e, b0 + step))), dtype=np.float64).reshape(-1, width)
             for b0 in range(s, e, step)]
    local = np.concatenate(parts, axis=0) if parts else np.zeros((0, width))
    return dict(records=gather_records(local, blocks, device=device, width=width), blocks=blocks)


def _device_posteriors(model, samples, prior, params, quantiles, log_nhi_threshold):
    """The CUDA path of one rank: spectra -> process_device -> posteriors_device -> host records."""
    import os
    import torch
    from .api import DLAProcessor, pad_spectra
    from .params import DEFAULT
    dev = int(os.environ.get("LOCAL_RANK", 0))
    proc = DLAProcessor(model, samples, prior, params or DEFAULT, device=dev)

    def compute(sp):
        pad = pad_spectra(sp)
        d = torch.device("cuda", dev)
        up = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dtype=dt)).to(d)
        out = proc.process_device(up(pad["wavelengths"], np.float64), up(pad["flux"], np.float64),
                                  up(pad["noise_variance"], np.float64), up(pad["pixel_mask"], np.uint8),
                                  up(pad["lengths"], np.int32), up(pad["z_qsos"], np.float64),
                                  return_sample_log_likelihoods=True)
        return proc.posteriors_device(out, quantiles, log_nhi_threshold).cpu().numpy()
    return compute


def multi_dla_posteriors_sharded(model: Dict, samples: Dict, spectra: Dict, prior: Dict, quantiles=None,
                                 log_nhi_threshold: float = None, params=None, max_dlas: int = 4,
                                 batch_quasars: int = 4096,
                                 compute: Callable[[Dict], Tuple[np.ndarray, np.ndarray]] = None,
                                 device=None) -> Dict:
    """``dla_posteriors_sharded`` for the multi-DLA model: rank r runs its cost-balanced block through
    ``process_multi_device`` (up to ``max_dlas`` DLAs, sub-DLA model, mean flux; ``samples`` holds the sub-DLA samples)
    in batches, then ``multi_posteriors_device`` and ``multi_posterior_quantiles_device``; one ``all_gather`` carries
    both records of every quasar side by side.  ``compute(spectra) -> (records, quantile_records)`` replaces the CUDA
    path of one rank.  Returns ``records`` [Q x (J + 2 J (J + 1))] (``api.unpack_multi_dla_posteriors``),
    ``quantile_records`` [Q x J (J + 1) / 2 (1 + 2 P)] (``api.unpack_multi_dla_posterior_quantiles``), both in
    catalogue order, and ``blocks``."""
    import torch.distributed as dist
    from . import params as P
    from .api import DEFAULT_QUANTILES, multi_dla_posterior_quantiles_width, multi_dla_posteriors_width
    quantiles = np.asarray(DEFAULT_QUANTILES if quantiles is None else quantiles, dtype=np.float64).ravel()
    log_nhi_threshold = P.dla_log_nhi_min if log_nhi_threshold is None else log_nhi_threshold
    rank, world = dist.get_rank(), dist.get_world_size()
    blocks = partition_by_cost(quasar_costs(spectra), world)
    s, e = blocks[rank]
    w0, w1 = multi_dla_posteriors_width(max_dlas), multi_dla_posterior_quantiles_width(max_dlas, quantiles.size)
    if compute is None and e > s:
        compute = _device_multi_posteriors(model, samples, prior, params, max_dlas, quantiles, log_nhi_threshold)
    step = max(int(batch_quasars), 1)
    parts = []
    for b0 in range(s, e, step):
        rec, qrec = compute(slice_spectra(spectra, b0, min(e, b0 + step)))
        parts.append(np.concatenate([np.asarray(rec, dtype=np.float64).reshape(-1, w0),
                                     np.asarray(qrec, dtype=np.float64).reshape(-1, w1)], axis=1))
    local = np.concatenate(parts, axis=0) if parts else np.zeros((0, w0 + w1))
    both = gather_records(local, blocks, device=device, width=w0 + w1)
    return dict(records=both[:, :w0].copy(), quantile_records=both[:, w0:].copy(), blocks=blocks)


def _device_multi_posteriors(model, samples, prior, params, max_dlas, quantiles, log_nhi_threshold):
    """The CUDA path of one rank: spectra -> process_multi_device -> multi_posteriors_device and
    multi_posterior_quantiles_device -> host records."""
    import os
    import torch
    from .api import DLAProcessor, pad_spectra
    from .params import DEFAULT
    dev = int(os.environ.get("LOCAL_RANK", 0))
    proc = DLAProcessor(model, samples, prior, params or DEFAULT, device=dev)

    def compute(sp):
        pad = pad_spectra(sp)
        d = torch.device("cuda", dev)
        up = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dtype=dt)).to(d)
        out = proc.process_multi_device(up(pad["wavelengths"], np.float64), up(pad["flux"], np.float64),
                                        up(pad["noise_variance"], np.float64), up(pad["pixel_mask"], np.uint8),
                                        up(pad["lengths"], np.int32), up(pad["z_qsos"], np.float64),
                                        max_dlas=max_dlas, return_samples=True)
        return (proc.multi_posteriors_device(out).cpu().numpy(),
                proc.multi_posterior_quantiles_device(out, quantiles, log_nhi_threshold).cpu().numpy())
    return compute
