"""Host-side mirror of the reference's interface for the hot path.

``process_qsos`` takes what the MATLAB script ``process_qsos.m`` reads from its ``.mat`` inputs
(process_qsos.m:4-49) and returns the variables it saves (process_qsos.m:236-244) with the
same names and shapes, plus ``map_z_dlas`` / ``map_log_nhis`` / ``map_inds``
(generate_ascii_catalog.m:73-80).  ``voigt`` mirrors the MEX signature
``profile = voigt(lambdas, z, N [, num_lines])`` (voigt.c:8-13,253-304; default 31 lines).

All compute happens in libgpdla.so (hand-written sm_100a CUDA) through the C ABI of
``include/gpdla.h``.  PyTorch is used only for device buffers and streams in the
device-resident entry points.  There is no CPU fallback.
"""
from __future__ import annotations

import ctypes
from typing import Dict, Optional, Sequence

import numpy as np

from . import _lib
from . import params as _params
from .params import DEFAULT, MULTI, Parameters, lya_wavelength

RESULT_NAMES = ["min_z_dlas", "max_z_dlas", "log_priors_no_dla", "log_priors_dla", "log_likelihoods_no_dla",
                "log_likelihoods_dla", "log_posteriors_no_dla", "log_posteriors_dla", "model_posteriors",
                "p_no_dlas", "p_dlas", "map_z_dlas", "map_log_nhis"]


def _f64(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.float64)


def _dp(a: np.ndarray):
    return a.ctypes.data_as(_lib.c_double_p)


def pad_spectra(spectra: Dict) -> Dict[str, np.ndarray]:
    """Ragged cell arrays (preload_qsos.m:73-79) -> padded ``[Q x L_max]`` planes + lengths."""
    if "lengths" in spectra:
        return spectra
    W = spectra["all_wavelengths"]
    Q = len(W)
    lengths = np.array([len(w) for w in W], dtype=np.int32)
    L_max = max(int(lengths.max()) if Q else 1, 1)
    out = dict(wavelengths=np.zeros((Q, L_max)), flux=np.zeros((Q, L_max)),
               noise_variance=np.ones((Q, L_max)), pixel_mask=np.ones((Q, L_max), dtype=np.uint8),
               lengths=lengths, z_qsos=_f64(spectra["z_qsos"]))
    for q in range(Q):
        n = lengths[q]
        out["wavelengths"][q, :n] = spectra["all_wavelengths"][q]
        out["flux"][q, :n] = spectra["all_flux"][q]
        out["noise_variance"][q, :n] = spectra["all_noise_variance"][q]
        out["pixel_mask"][q, :n] = np.asarray(spectra["all_pixel_mask"][q]).astype(np.uint8)
    return out


def _check_planes(W, F, V, Mk, lengths, z):
    """The padded planes must share one [Q x L_max] shape and every length must fit its row."""
    if W.ndim != 2 or F.shape != W.shape or V.shape != W.shape or Mk.shape != W.shape:
        raise ValueError("wavelengths, flux, noise_variance and pixel_mask must share one (Q, L_max) shape")
    if lengths.shape != (W.shape[0],) or z.shape != (W.shape[0],):
        raise ValueError("lengths and z_qsos must have one entry per quasar")
    if lengths.size and (lengths.min() < 0 or lengths.max() > W.shape[1]):
        raise ValueError("lengths must lie in [0, L_max]")


class DLAProcessor:
    """A libgpdla context holding the learned null model, the DLA samples and the prior
    catalogue on one GPU (what process_qsos.m:4-40 loads once before its quasar loop)."""

    def __init__(self, model: Dict, samples: Dict, prior: Dict, params: Parameters = DEFAULT, device: int = 0,
                 batch_quasars: int = 0, gram_digits: int = 0, rest_table: int = 0):
        """``gram_digits``: arithmetic of the Gram contraction -- 0 default (exact-product INT8 tensor-core path
        with 6 digits for k = 20 and 40, FP64 DMMA for k = 10), -1 FP64 DMMA, 5 / 6 INT8 path with that many digits (k = 40: 6).
        ``rest_table``: 0 default (optical depth from the rest-frame table away from the line centres), -1 direct
        evaluation of the line sum everywhere (``gpdla_params.rest_table``)."""
        self._lib = _lib.load()
        self._pinned = {}
        self._ctx = ctypes.c_void_p()
        _lib.check(self._lib.gpdla_create(ctypes.byref(self._ctx), int(device)))
        self.device = int(device)
        self.params = params
        p = _lib.GpdlaParams()
        self._lib.gpdla_default_parameters(ctypes.byref(p))
        p.min_lambda, p.max_lambda = params.min_lambda, params.max_lambda
        p.prior_z_qso_increase = params.prior_z_qso_increase
        p.min_z_cut, p.max_z_cut = params.min_z_cut, params.max_z_cut
        p.pixel_spacing, p.num_lines, p.batch_quasars = params.pixel_spacing, params.num_lines, int(batch_quasars)
        p.gram_digits = int(gram_digits)
        p.rest_table = int(rest_table)
        _lib.check(self._lib.gpdla_set_parameters(self._ctx, ctypes.byref(p)), self._ctx)
        rest, mu, M, lw = (_f64(model[k]) for k in ("rest_wavelengths", "mu", "M", "log_omega"))
        if M.shape != (rest.size, M.shape[1]) or mu.size != rest.size or lw.size != rest.size:
            raise ValueError("model arrays must be rest_wavelengths (n,), mu (n,), M (n, k), log_omega (n,)")
        self.k = int(M.shape[1])
        _lib.check(self._lib.gpdla_set_model(self._ctx, _dp(rest), rest.size, _dp(mu), _dp(M), self.k, _dp(lw),
                                             float(model["log_c_0"]), float(model["log_tau_0"]),
                                             float(model["log_beta"])), self._ctx)
        off, lnhi, nhi = (_f64(samples[k]).ravel() for k in ("offset_samples", "log_nhi_samples", "nhi_samples"))
        self.num_dla_samples = int(off.size)
        self._samples_host = (off, lnhi, nhi)
        self._samples_device = None          # CUDA copies for statistics_device, made on its first call
        _lib.check(self._lib.gpdla_set_samples(self._ctx, _dp(off), _dp(lnhi), _dp(nhi), off.size), self._ctx)
        self.has_lls = "lls_nhi_samples" in samples and "Z_lls" in samples and "Z_dla" in samples
        if self.has_lls:   # multi_dlas/set_lls_parameters.m:55-71
            lls = _f64(samples["lls_nhi_samples"]).ravel()
            _lib.check(self._lib.gpdla_set_lls_samples(self._ctx, _dp(lls), lls.size, float(samples["Z_lls"]),
                                                       float(samples["Z_dla"])), self._ctx)
        pz = _f64(prior["z_qsos"]).ravel()
        pd = np.ascontiguousarray(np.asarray(prior["dla_ind"]).astype(np.uint8)).ravel()
        _lib.check(self._lib.gpdla_set_prior(self._ctx, _dp(pz), pd.ctypes.data_as(_lib.c_u8_p), pz.size), self._ctx)

    def close(self):
        if getattr(self, "_ctx", None) is not None and self._ctx:
            self._lib.gpdla_destroy(self._ctx)
            self._ctx = ctypes.c_void_p()
        for ptr, _ in getattr(self, "_pinned", {}).values():
            self._lib.gpdla_host_free(ptr)
        self._pinned = {}

    def _pinned_array(self, name: str, shape, dtype=np.float64) -> np.ndarray:
        """A page-locked host array owned by this processor (``gpdla_host_alloc``), reused while the shape
        holds: result copies into it overlap the next batch's kernels.  Valid until the next call / ``close``."""
        nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
        have = self._pinned.get(name)
        if have is None or have[1] < nbytes:
            if have is not None:
                self._lib.gpdla_host_free(have[0])
            ptr = ctypes.c_void_p()
            _lib.check(self._lib.gpdla_host_alloc(ctypes.byref(ptr), max(nbytes, 1)))
            self._pinned[name] = have = (ptr, nbytes)
        buf = (ctypes.c_char * max(nbytes, 1)).from_address(have[0].value)
        return np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def launch_count(self) -> int:
        return int(self._lib.gpdla_launch_count(self._ctx))

    def set_profiling(self, enable: bool):
        _lib.check(self._lib.gpdla_set_profiling(self._ctx, int(bool(enable))), self._ctx)

    def profile_read(self):
        """(summed ms, launches) of the fused log-likelihood kernel since the last read."""
        ms, n = ctypes.c_double(), ctypes.c_int64()
        _lib.check(self._lib.gpdla_profile_read(self._ctx, ctypes.byref(ms), ctypes.byref(n)), self._ctx)
        return ms.value, n.value

    # ---------------------------------------------------------------- host buffers (the drop-in call)
    def process(self, spectra: Dict, return_sample_log_likelihoods: bool = True,
                pinned_results: bool = False) -> Dict[str, np.ndarray]:
        """The body of process_qsos.m for the given spectra (host arrays in, host arrays out).
        ``pinned_results``: ``sample_log_likelihoods_dla`` (80 KB per quasar) is returned in a page-locked buffer
        owned by this processor -- valid until the next ``process`` call -- so that its copy overlaps compute."""
        sp = pad_spectra(spectra)
        W, F, V = _f64(sp["wavelengths"]), _f64(sp["flux"]), _f64(sp["noise_variance"])
        Mk = np.ascontiguousarray(sp["pixel_mask"], dtype=np.uint8)
        lengths = np.ascontiguousarray(sp["lengths"], dtype=np.int32).ravel()
        z = _f64(sp["z_qsos"]).ravel()
        _check_planes(W, F, V, Mk, lengths, z)
        Q, L_max = W.shape
        S = self.num_dla_samples
        out = {n: np.full((Q, 2) if n == "model_posteriors" else (Q,), np.nan) for n in RESULT_NAMES}
        out["map_inds"] = np.full(Q, -1, dtype=np.int64)
        if return_sample_log_likelihoods:
            if pinned_results:
                out["sample_log_likelihoods_dla"] = self._pinned_array("sll", (Q, S))
                out["sample_log_likelihoods_dla"].fill(np.nan)
            else:
                out["sample_log_likelihoods_dla"] = np.full((Q, S), np.nan)
        res = _lib.GpdlaResults()
        for n in _lib.RESULT_F64:
            setattr(res, n, out[n].ctypes.data if n in out else None)
        res.map_inds = out["map_inds"].ctypes.data
        vp = lambda a: ctypes.c_void_p(a.ctypes.data)
        _lib.check(self._lib.gpdla_process_qsos(self._ctx, Q, L_max, vp(W), vp(F), vp(V), vp(Mk), vp(lengths),
                                                vp(z), ctypes.byref(res)), self._ctx)
        return out

    # ---------------------------------------------------------------- multi-DLA + sub-DLA + mean flux
    def process_multi(self, spectra: Dict, max_dlas: int = 4, base_sample_inds: Optional[np.ndarray] = None,
                      return_samples: bool = True) -> Dict[str, np.ndarray]:
        """``process_qsos_multiple_dlas_meanflux`` (multi_dlas/process_qsos_multiple_dlas_meanflux.m): results
        with the reference's names and shapes -- ``sample_log_likelihoods_dla`` (Q, S, max_dlas),
        ``base_sample_inds`` (Q, S, max_dlas-1; 0-based), ``MAP_*`` (Q, max_dlas, max_dlas),
        ``model_posteriors`` (Q, 2 + max_dlas).  ``base_sample_inds`` given as input (same shape) replaces
        the built-in resampling (rng('default') + randsample) for parity runs."""
        if not self.has_lls:
            raise ValueError("samples must hold lls_nhi_samples, Z_lls and Z_dla for the multi-DLA path")
        sp = pad_spectra(spectra)
        W, F, V = _f64(sp["wavelengths"]), _f64(sp["flux"]), _f64(sp["noise_variance"])
        Mk = np.ascontiguousarray(sp["pixel_mask"], dtype=np.uint8)
        lengths = np.ascontiguousarray(sp["lengths"], dtype=np.int32).ravel()
        z = _f64(sp["z_qsos"]).ravel()
        _check_planes(W, F, V, Mk, lengths, z)
        Q, L_max = W.shape
        S, MD = self.num_dla_samples, int(max_dlas)
        shapes = dict(log_priors_dla=(Q, MD), log_likelihoods_dla=(Q, MD), log_posteriors_dla=(Q, MD),
                      model_posteriors=(Q, MD + 2), MAP_z_dlas=(Q, MD, MD), MAP_log_nhis=(Q, MD, MD))
        out = {}
        for n in _lib.MULTI_RESULT_FIELDS[:17]:
            out[n] = np.full(shapes.get(n, (Q,)), np.nan)
        out["MAP_inds"] = np.full((Q, MD, MD), -1, dtype=np.int64)
        if return_samples:
            out["sample_log_likelihoods_dla"] = np.full((Q, MD, S), np.nan)
            out["sample_log_likelihoods_lls"] = np.full((Q, S), np.nan)
            out["base_sample_inds"] = np.zeros((Q, max(MD - 1, 0), S), dtype=np.int32)
        res = _lib.GpdlaMultiResults()
        for n in _lib.MULTI_RESULT_FIELDS:
            setattr(res, n, out[n].ctypes.data if n in out and out[n].size else None)
        bin_ = None
        if base_sample_inds is not None:
            bin_ = np.ascontiguousarray(np.transpose(np.asarray(base_sample_inds), (0, 2, 1)), dtype=np.int32)
            assert bin_.shape == (Q, MD - 1, S)
        vp = lambda a: ctypes.c_void_p(a.ctypes.data)
        _lib.check(self._lib.gpdla_process_qsos_multi(
            self._ctx, Q, L_max, vp(W), vp(F), vp(V), vp(Mk), vp(lengths), vp(z), MD,
            vp(bin_) if bin_ is not None else None, ctypes.byref(res)), self._ctx)
        if return_samples:   # reference layout: (quasar, sample, level)
            out["sample_log_likelihoods_dla"] = np.transpose(out["sample_log_likelihoods_dla"], (0, 2, 1))
            out["base_sample_inds"] = np.transpose(out["base_sample_inds"], (0, 2, 1))
        return out

    # ---------------------------------------------------------------- device-resident buffers
    def process_device(self, wavelengths, flux, noise_variance, pixel_mask, lengths, z_qsos,
                       return_sample_log_likelihoods: bool = False, out: Optional[Dict] = None) -> Dict:
        """Inputs are CUDA tensors (float64 [Q x L_max], uint8 mask, int32 lengths, float64 z);
        returns CUDA tensors.  Asynchronous on torch's current stream."""
        import torch
        Q, L_max = wavelengths.shape
        dev = wavelengths.device
        assert dev.type == "cuda" and dev.index == self.device
        for t, dt in ((wavelengths, torch.float64), (flux, torch.float64), (noise_variance, torch.float64),
                      (pixel_mask, torch.uint8), (lengths, torch.int32), (z_qsos, torch.float64)):
            assert t.is_cuda and t.dtype == dt and t.is_contiguous()
        if out is None:
            out = {n: torch.empty((Q, 2) if n == "model_posteriors" else (Q,), dtype=torch.float64, device=dev)
                   for n in RESULT_NAMES}
            out["map_inds"] = torch.empty(Q, dtype=torch.int64, device=dev)
            if return_sample_log_likelihoods:
                out["sample_log_likelihoods_dla"] = torch.empty((Q, self.num_dla_samples), dtype=torch.float64,
                                                                device=dev)
        res = _lib.GpdlaResults()
        for n in _lib.RESULT_F64:
            setattr(res, n, out[n].data_ptr() if n in out else None)
        res.map_inds = out["map_inds"].data_ptr()
        stream = torch.cuda.current_stream(dev).cuda_stream
        _lib.check(self._lib.gpdla_process_qsos_device(
            self._ctx, Q, L_max, wavelengths.data_ptr(), flux.data_ptr(), noise_variance.data_ptr(),
            pixel_mask.data_ptr(), lengths.data_ptr(), z_qsos.data_ptr(), ctypes.byref(res),
            ctypes.c_void_p(stream)), self._ctx)
        return out

    def process_multi_device(self, wavelengths, flux, noise_variance, pixel_mask, lengths, z_qsos, max_dlas: int = 4,
                             base_sample_inds=None, return_samples: bool = False, out: Optional[Dict] = None) -> Dict:
        """The device-resident twin of ``process_multi``: inputs as ``process_device`` takes them, CUDA tensors out, in
        the C layout -- ``model_posteriors`` [Q, 2 + max_dlas], ``MAP_*`` [Q, max_dlas, max_dlas] and, with
        ``return_samples``, ``sample_log_likelihoods_dla`` [Q, max_dlas, S], ``sample_log_likelihoods_lls`` [Q, S] and
        ``base_sample_inds`` [Q, max_dlas - 1, S] (int32, 0-based).  ``base_sample_inds`` given as input (an int32 CUDA
        tensor [Q, max_dlas - 1, S]) replaces the built-in resampling.  Asynchronous on torch's current stream."""
        import torch
        if not self.has_lls:
            raise ValueError("samples must hold lls_nhi_samples, Z_lls and Z_dla for the multi-DLA path")
        MD = int(max_dlas)
        if not 1 <= MD <= 4:
            raise ValueError("max_dlas must lie in [1, 4]")
        Q, L_max = wavelengths.shape
        dev = wavelengths.device
        assert dev.type == "cuda" and dev.index == self.device
        for t, dt in ((wavelengths, torch.float64), (flux, torch.float64), (noise_variance, torch.float64),
                      (pixel_mask, torch.uint8), (lengths, torch.int32), (z_qsos, torch.float64)):
            assert t.is_cuda and t.dtype == dt and t.is_contiguous()
        S = self.num_dla_samples
        if out is None:
            shapes = dict(log_priors_dla=(Q, MD), log_likelihoods_dla=(Q, MD), log_posteriors_dla=(Q, MD),
                          model_posteriors=(Q, MD + 2), MAP_z_dlas=(Q, MD, MD), MAP_log_nhis=(Q, MD, MD))
            out = {n: torch.empty(shapes.get(n, (Q,)), dtype=torch.float64, device=dev)
                   for n in _lib.MULTI_RESULT_FIELDS[:17]}
            out["MAP_inds"] = torch.empty((Q, MD, MD), dtype=torch.int64, device=dev)
            if return_samples:
                out["sample_log_likelihoods_dla"] = torch.full((Q, MD, S), float("nan"), dtype=torch.float64, device=dev)
                out["sample_log_likelihoods_lls"] = torch.full((Q, S), float("nan"), dtype=torch.float64, device=dev)
                out["base_sample_inds"] = torch.zeros((Q, MD - 1, S), dtype=torch.int32, device=dev)
        res = _lib.GpdlaMultiResults()
        for n in _lib.MULTI_RESULT_FIELDS:
            setattr(res, n, out[n].data_ptr() if n in out and out[n].numel() else None)
        bin_ = None
        if base_sample_inds is not None and MD > 1:
            if not (base_sample_inds.is_cuda and base_sample_inds.dtype == torch.int32
                    and tuple(base_sample_inds.shape) == (Q, MD - 1, S)):
                raise ValueError("base_sample_inds must be an int32 CUDA tensor [Q, max_dlas - 1, S]")
            # the device entry reads given indices with a stride of 3 S per quasar, as its workspace holds them
            bin_ = torch.zeros((Q, 3, S), dtype=torch.int32, device=dev)
            bin_[:, :MD - 1] = base_sample_inds
        stream = torch.cuda.current_stream(dev).cuda_stream
        _lib.check(self._lib.gpdla_process_qsos_multi_device(
            self._ctx, Q, L_max, wavelengths.data_ptr(), flux.data_ptr(), noise_variance.data_ptr(),
            pixel_mask.data_ptr(), lengths.data_ptr(), z_qsos.data_ptr(), MD,
            None if bin_ is None else bin_.data_ptr(), ctypes.byref(res), ctypes.c_void_p(stream)), self._ctx)
        return out

    def _stats_operands(self, dev, Q: int, S: int, width: int, select, sums):
        """Device samples (copied once), the sums tensor to add into and the uint8 select mask of a statistics call."""
        import torch
        if S != self.num_dla_samples:
            raise ValueError("sample_log_likelihoods_dla has %d samples, this processor %d" % (S, self.num_dla_samples))
        if self._samples_device is None:
            self._samples_device = tuple(torch.from_numpy(a).to(dev) for a in self._samples_host)
        if sums is None:
            sums = torch.zeros(width, dtype=torch.float64, device=dev)
        if not (sums.is_cuda and sums.device == dev and sums.dtype == torch.float64 and sums.is_contiguous()
                and sums.numel() == width):
            raise ValueError("sums must be a contiguous float64 CUDA tensor of %d entries on %s" % (width, dev))
        sel = None
        if select is not None:
            sel = select.to(device=dev, dtype=torch.uint8).contiguous()
            if sel.shape != (Q,):
                raise ValueError("select must have one entry per quasar")
        return self._samples_device, sums, sel

    def statistics_device(self, out: Dict, z_edges, log_nhi_edges, select=None, sums=None,
                          dla_log_nhi_min: float = _params.dla_log_nhi_min, omega_m: float = _params.omega_m):
        """Population-statistics sums (``dla_statistics_sums``) of what ``process_device(...,
        return_sample_log_likelihoods=True)`` returned, without the sample log-likelihoods leaving the GPU.  ``select``:
        optional CUDA bool / uint8 tensor [Q]; ``sums``: a float64 CUDA tensor to add into (a new zero vector when None).
        Returns the sums tensor; asynchronous on torch's current stream.  Uses device copies of this processor's samples,
        made once."""
        import torch
        ll = out.get("sample_log_likelihoods_dla")
        if ll is None:
            raise ValueError("statistics_device needs process_device(..., return_sample_log_likelihoods=True)")
        dev = ll.device
        Q, S = ll.shape
        ze, ne = _stats_edges(z_edges, log_nhi_edges)
        (off, lnhi, nhi), sums, sel = self._stats_operands(dev, Q, S, dla_statistics_width(ze.size - 1, ne.size - 1),
                                                           select, sums)
        ptr = lambda t: None if t is None else ctypes.c_void_p(t.data_ptr())
        with torch.cuda.device(dev):
            stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
            _lib.check(self._lib.gpdla_dla_statistics_device(
                Q, S, ptr(ll), ptr(out["p_dlas"]), ptr(out["min_z_dlas"]), ptr(out["max_z_dlas"]), ptr(sel), ptr(off),
                ptr(lnhi), ptr(nhi), ze.size - 1, _dp(ze), ne.size - 1, _dp(ne), float(dla_log_nhi_min),
                float(omega_m), ptr(sums), stream))
        return sums

    def multi_statistics_device(self, out: Dict, z_edges, log_nhi_edges, select=None, sums=None,
                                dla_log_nhi_min: float = _params.dla_log_nhi_min, omega_m: float = _params.omega_m):
        """Population-statistics sums of the multi-DLA model (``multi_dla_statistics_sums``) of what
        ``process_multi_device(..., return_samples=True)`` returned, without the per-sample arrays leaving the GPU.
        ``select``: optional CUDA bool / uint8 tensor [Q]; ``sums``: a float64 CUDA tensor to add into (a new zero
        vector when None).  Returns the sums tensor; asynchronous on torch's current stream.  Uses device copies of this
        processor's samples, made once."""
        import torch
        ll = out.get("sample_log_likelihoods_dla")
        if ll is None:
            raise ValueError("multi_statistics_device needs process_multi_device(..., return_samples=True)")
        dev = ll.device
        Q, J, S = ll.shape
        part = out.get("base_sample_inds")
        if J > 1 and (part is None or tuple(part.shape) != (Q, J - 1, S) or part.dtype != torch.int32
                      or not part.is_contiguous()):
            raise ValueError("base_sample_inds must be a contiguous int32 tensor [Q, max_dlas - 1, S]")
        if tuple(out["model_posteriors"].shape) != (Q, J + 2):
            raise ValueError("model_posteriors must be [Q, 2 + max_dlas]")
        if not all(out[n].is_contiguous() for n in ("sample_log_likelihoods_dla", "model_posteriors", "min_z_dlas",
                                                    "max_z_dlas")):
            raise ValueError("the arrays of process_multi_device must be contiguous")
        ze, ne = _stats_edges(z_edges, log_nhi_edges)
        (off, lnhi, nhi), sums, sel = self._stats_operands(dev, Q, S, dla_statistics_width(ze.size - 1, ne.size - 1),
                                                           select, sums)
        ptr = lambda t: None if t is None else ctypes.c_void_p(t.data_ptr())
        with torch.cuda.device(dev):
            stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
            _lib.check(self._lib.gpdla_multi_dla_statistics_device(
                Q, S, J, ptr(ll), ptr(part if J > 1 else None), ptr(out["model_posteriors"]), ptr(out["min_z_dlas"]), ptr(out["max_z_dlas"]), ptr(sel),
                ptr(off), ptr(lnhi), ptr(nhi), ze.size - 1, _dp(ze), ne.size - 1, _dp(ne), float(dla_log_nhi_min),
                float(omega_m), ptr(sums), stream))
        return sums

    # ---------------------------------------------------------------- fitted model under chosen absorbers
    def _recon_operands(self, Q: int, absorber_z, absorber_nhi, to):
        """(num_absorbers, z, N) as [Q x num_absorbers] arrays made by ``to`` (NaN z = no absorber)."""
        if (absorber_z is None) != (absorber_nhi is None):
            raise ValueError("absorber_z and absorber_nhi go together")
        if absorber_z is None:
            return 0, None, None
        z, n = to(absorber_z), to(absorber_nhi)
        if z.ndim == 1:
            z, n = z.reshape(-1, 1), n.reshape(-1, 1)
        if tuple(z.shape) != tuple(n.shape) or z.ndim != 2 or z.shape[0] != Q or not 0 <= z.shape[1] <= 4:
            raise ValueError("absorber_z and absorber_nhi must be [Q, num_absorbers] with 0 <= num_absorbers <= 4")
        return int(z.shape[1]), z, n

    def reconstruct(self, spectra: Dict, absorber_z=None, absorber_nhi=None, meanflux: bool = False) -> Dict[str, np.ndarray]:
        """The model fitted to each spectrum under the given absorbers (``gpdla_reconstruct``; what
        CDDF_analysis/qso_loader.py:1654-1774 draws).  ``spectra``: ragged or padded, as ``process`` takes them;
        ``absorber_z`` / ``absorber_nhi``: [Q, num_absorbers] (0..4; N in cm^-2; NaN z = none) or None for the null
        model; ``meanflux``: the multi-DLA path's null model.  Returns NumPy arrays: the planes ``absorption``,
        ``prior_mean``, ``prior_sd``, ``fit_mean``, ``continuum``, ``continuum_sd`` [Q, L_max] on each quasar's own
        pixels (``wavelengths[q, :lengths[q]]``; NaN outside the modelled window), ``latent`` [Q, k], ``chi2``,
        ``log_likelihood`` and ``num_pixels`` [Q]."""
        sp = pad_spectra(spectra)
        W, F, V = _f64(sp["wavelengths"]), _f64(sp["flux"]), _f64(sp["noise_variance"])
        Mk = np.ascontiguousarray(sp["pixel_mask"], dtype=np.uint8)
        lengths = np.ascontiguousarray(sp["lengths"], dtype=np.int32).ravel()
        z = _f64(sp["z_qsos"]).ravel()
        _check_planes(W, F, V, Mk, lengths, z)
        Q, L_max = W.shape
        A, az, an = self._recon_operands(Q, absorber_z, absorber_nhi, _f64)
        out = {n: np.empty((Q, L_max)) for n in _lib.RECONSTRUCTION_FIELDS[:6]}
        out.update(latent=np.empty((Q, self.k)), chi2=np.empty(Q), log_likelihood=np.empty(Q),
                   num_pixels=np.empty(Q, dtype=np.int32))
        res = _lib.GpdlaReconstruction()
        for n in _lib.RECONSTRUCTION_FIELDS:
            setattr(res, n, out[n].ctypes.data if out[n].size else None)
        vp = lambda a: None if a is None else ctypes.c_void_p(a.ctypes.data)
        _lib.check(self._lib.gpdla_reconstruct(self._ctx, Q, L_max, vp(W), vp(F), vp(V), vp(Mk), vp(lengths), vp(z),
                                               int(bool(meanflux)), A, vp(az), vp(an), ctypes.byref(res)), self._ctx)
        return out

    def reconstruct_device(self, wavelengths, flux, noise_variance, pixel_mask, lengths, z_qsos, absorber_z=None,
                           absorber_nhi=None, meanflux: bool = False) -> Dict:
        """Device-resident ``reconstruct``: the planes as ``process_device`` (and ``preload_qsos_device``) hold them,
        absorbers as CUDA tensors or host arrays; returns CUDA tensors with the names of ``reconstruct``.  Asynchronous
        on torch's current stream."""
        import torch
        Q, L_max = wavelengths.shape
        dev = wavelengths.device
        assert dev.type == "cuda" and dev.index == self.device
        for t, dt in ((wavelengths, torch.float64), (flux, torch.float64), (noise_variance, torch.float64),
                      (pixel_mask, torch.uint8), (lengths, torch.int32), (z_qsos, torch.float64)):
            assert t.is_cuda and t.dtype == dt and t.is_contiguous()
        to = lambda a: torch.as_tensor(a, dtype=torch.float64, device=dev).contiguous()
        A, az, an = self._recon_operands(Q, absorber_z, absorber_nhi, to)
        f64 = dict(dtype=torch.float64, device=dev)
        out = {n: torch.empty((Q, L_max), **f64) for n in _lib.RECONSTRUCTION_FIELDS[:6]}
        out.update(latent=torch.empty((Q, self.k), **f64), chi2=torch.empty(Q, **f64),
                   log_likelihood=torch.empty(Q, **f64), num_pixels=torch.empty(Q, dtype=torch.int32, device=dev))
        res = _lib.GpdlaReconstruction()
        for n in _lib.RECONSTRUCTION_FIELDS:
            setattr(res, n, out[n].data_ptr() if out[n].numel() else None)
        ptr = lambda t: None if t is None else ctypes.c_void_p(t.data_ptr())
        stream = torch.cuda.current_stream(dev).cuda_stream
        _lib.check(self._lib.gpdla_reconstruct_device(
            self._ctx, Q, L_max, ptr(wavelengths), ptr(flux), ptr(noise_variance), ptr(pixel_mask), ptr(lengths),
            ptr(z_qsos), int(bool(meanflux)), A, ptr(az if A else None), ptr(an if A else None), ctypes.byref(res),
            ctypes.c_void_p(stream)), self._ctx)
        return out


def process_qsos(model: Dict, samples: Dict, spectra: Dict, prior: Dict, params: Parameters = DEFAULT,
                 device: int = 0, return_sample_log_likelihoods: bool = True, gram_digits: int = 0,
                 rest_table: int = 0) -> Dict[str, np.ndarray]:
    """Run the DLA detection algorithm on the given objects (process_qsos.m)."""
    proc = DLAProcessor(model, samples, prior, params, device, gram_digits=gram_digits, rest_table=rest_table)
    try:
        return proc.process(spectra, return_sample_log_likelihoods)
    finally:
        proc.close()


def process_qsos_multiple_dlas_meanflux(model: Dict, samples: Dict, spectra: Dict, prior: Dict, max_dlas: int = 4,
                                        params: Parameters = DEFAULT, device: int = 0,
                                        base_sample_inds: Optional[np.ndarray] = None,
                                        return_samples: bool = True, batch_quasars: int = 0,
                                        gram_digits: int = 0, rest_table: int = 0) -> Dict[str, np.ndarray]:
    """Multi-DLA / sub-DLA / mean-flux processing (multi_dlas/process_qsos_multiple_dlas_meanflux.m).
    ``samples`` additionally holds ``lls_nhi_samples``, ``Z_lls``, ``Z_dla`` (set_lls_parameters.m)."""
    proc = DLAProcessor(model, samples, prior, params, device, batch_quasars=batch_quasars, gram_digits=gram_digits,
                        rest_table=rest_table)
    try:
        return proc.process_multi(spectra, max_dlas, base_sample_inds, return_samples)
    finally:
        proc.close()


def _host(a) -> np.ndarray:
    """A result array on the host (NumPy as it is; CUDA tensors copied)."""
    if hasattr(a, "detach"):
        a = a.detach().cpu().numpy()
    return np.asarray(a)


def map_absorbers(results: Dict, samples: Dict, model="map"):
    """The absorbers of one model of a processed batch, as ``DLAProcessor.reconstruct`` takes them:
    ``(absorber_z, absorber_nhi)``, [Q, num_absorbers] NumPy arrays (NaN z = none).  ``results``: what ``process``,
    ``process_device``, ``process_multi(_device)`` or ``process_qsos_multiple_dlas_meanflux`` returned; ``samples``:
    the samples they ran with.  ``model``:

    * ``"map"``: each quasar's most probable model by ``model_posteriors`` (single-DLA: ``p_dlas > p_no_dlas``);
    * ``"null"``: no absorbers;
    * an integer j: level j's MAP absorbers, z from ``MAP_z_dlas`` (``map_z_dlas``) and N = ``nhi_samples[MAP_inds]``
      (the sample's own N, not ``10**MAP_log_nhis``), so the reconstruction's log-likelihood is the stored sample's;
    * ``"sub_dla"``: the arg-max of ``sample_log_likelihoods_lls`` at its (z_i, ``lls_nhi_samples[i]``)."""
    nhi = _f64(samples["nhi_samples"]).ravel()
    multi = "MAP_z_dlas" in results
    Q = _host(results["min_z_dlas"]).shape[0]
    none = lambda A: (np.full((Q, A), np.nan), np.full((Q, A), np.nan))

    def level(j):
        if multi:
            MD = _host(results["MAP_z_dlas"]).shape[1]
            if not 1 <= j <= MD:
                raise ValueError("level must lie in [1, %d]" % MD)
            zz = _host(results["MAP_z_dlas"])[:, j - 1, :j].astype(np.float64)
            ind = _host(results["MAP_inds"])[:, j - 1, :j].astype(np.int64)
        else:
            if j != 1:
                raise ValueError("single-DLA results hold level 1 only")
            zz = _host(results["map_z_dlas"]).astype(np.float64).reshape(Q, 1)
            ind = _host(results["map_inds"]).astype(np.int64).reshape(Q, 1)
        ok = ind >= 0
        n = np.where(ok, nhi[np.where(ok, ind, 0)], np.nan)
        return np.where(ok, zz, np.nan), n

    def sub_dla():
        if "sample_log_likelihoods_lls" not in results or "lls_nhi_samples" not in samples:
            raise ValueError('model="sub_dla" needs results["sample_log_likelihoods_lls"] (process_multi with '
                             'return_samples) and samples["lls_nhi_samples"]')
        ll = _host(results["sample_log_likelihoods_lls"])
        lls = _f64(samples["lls_nhi_samples"]).ravel()
        off = _f64(samples["offset_samples"]).ravel()
        zlo, zhi = _host(results["min_z_dlas"]), _host(results["max_z_dlas"])
        zz, n = none(1)
        for q in range(Q):
            if np.all(np.isnan(ll[q])):
                continue
            i = int(np.nanargmax(ll[q]))
            zz[q, 0] = zlo[q] + (zhi[q] - zlo[q]) * off[i]
            n[q, 0] = lls[i]
        return zz, n

    if isinstance(model, str) and model == "null":
        return none(0)
    if isinstance(model, str) and model == "sub_dla":
        if not multi:
            raise ValueError('model="sub_dla" needs multi-DLA results')
        return sub_dla()
    if isinstance(model, (int, np.integer)) and not isinstance(model, bool):
        return level(int(model))
    if not (isinstance(model, str) and model == "map"):
        raise ValueError('model must be "map", "null", "sub_dla" or a level number')
    if not multi:
        p_dla, p_no = _host(results["p_dlas"]), _host(results["p_no_dlas"])
        zz, n = level(1)
        dla = p_dla > p_no
        return np.where(dla[:, None], zz, np.nan), np.where(dla[:, None], n, np.nan)
    mp = _host(results["model_posteriors"])
    MD = mp.shape[1] - 2
    zz, n = none(MD)
    # NaN-ignoring arg-max (levels past an early exit are NaN); a row without a finite entry gets no absorber
    finite = np.any(np.isfinite(mp), axis=1)
    best = np.where(finite, np.argmax(np.where(np.isfinite(mp), mp, -np.inf), axis=1), 0)
    if np.any(best == 1):
        zs, ns = sub_dla()
        zz[best == 1, :1], n[best == 1, :1] = zs[best == 1], ns[best == 1]
    for j in range(1, MD + 1):
        sel = best == j + 1
        if np.any(sel):
            zj, nj = level(j)
            zz[sel, :j], n[sel, :j] = zj[sel], nj[sel]
    return zz, n


def _pad_raw(raw: Dict) -> Dict[str, np.ndarray]:
    F = raw["flux"]
    Q = len(F)
    lengths = np.array([len(f) for f in F], dtype=np.int32)
    L = max(int(lengths.max()) if Q else 1, 1)
    out = dict(flux=np.zeros((Q, L)), loglam=np.zeros((Q, L)), ivar=np.zeros((Q, L)),
               and_mask=np.zeros((Q, L), dtype=np.int32), lengths=lengths)
    for q in range(Q):
        n = lengths[q]
        out["flux"][q, :n] = raw["flux"][q]
        out["loglam"][q, :n] = raw["loglam"][q]
        out["ivar"][q, :n] = raw["ivar"][q]
        out["and_mask"][q, :n] = np.asarray(raw["and_mask"][q]).astype(np.int64).astype(np.int32)
    return out


def preload_qsos(raw: Dict, z_qsos, filter_flags=None, params: Parameters = DEFAULT, device: int = 0,
                 L_out: int = 0) -> Dict:
    """Spectrum preprocessing on the GPU: read_spec.m:28-38 + preload_qsos.m:18-71.

    ``raw`` holds the four columns of the SDSS speclite coadd table per quasar (ragged lists ``flux``, ``loglam``,
    ``ivar``, ``and_mask``; read_spec.m:11-26).  Returns the variables preload_qsos.m:73-79 saves --
    ``all_wavelengths``, ``all_flux``, ``all_noise_variance``, ``all_pixel_mask`` (ragged lists, empty for skipped
    quasars), ``all_normalizers`` -- and the updated ``filter_flags``; the dict can be passed to ``process_qsos``
    as ``spectra`` once ``z_qsos`` is added and the flagged quasars are dropped."""
    import torch
    lib = _lib.load()
    pad = _pad_raw(raw)
    Q, L_in = pad["flux"].shape
    z = _f64(z_qsos)
    if L_out <= 0:
        # the loading window spans log10(1217 / 910) / 1e-4 = 1263 pixels of the BOSS grid, + 2 edge pixels
        L_out = min(L_in, 1280)
    p = _lib.GpdlaPreloadParams()
    lib.gpdla_default_preload_parameters(ctypes.byref(p))
    p.min_lambda, p.max_lambda = params.min_lambda, params.max_lambda
    p.loading_min_lambda, p.loading_max_lambda = params.loading_min_lambda, params.loading_max_lambda
    p.min_num_pixels = params.min_num_pixels
    flags_in = None if filter_flags is None else np.ascontiguousarray(filter_flags, dtype=np.uint8)
    out = dict(wavelengths=np.zeros((Q, L_out)), flux=np.zeros((Q, L_out)), noise_variance=np.zeros((Q, L_out)),
               pixel_mask=np.zeros((Q, L_out), dtype=np.uint8), lengths=np.zeros(Q, dtype=np.int32),
               normalizers=np.zeros(Q), filter_flags=np.zeros(Q, dtype=np.uint8))
    vp = lambda a: None if a is None else a.ctypes.data_as(ctypes.c_void_p)
    with torch.cuda.device(device):
        _lib.check(lib.gpdla_preload_qsos(Q, L_in, vp(pad["flux"]), vp(pad["loglam"]), vp(pad["ivar"]), vp(pad["and_mask"]),
                                          vp(pad["lengths"]), vp(z), vp(flags_in), ctypes.byref(p), L_out,
                                          vp(out["wavelengths"]), vp(out["flux"]), vp(out["noise_variance"]),
                                          vp(out["pixel_mask"]), vp(out["lengths"]), vp(out["normalizers"]),
                                          vp(out["filter_flags"])))
    n = out["lengths"]
    return dict(all_wavelengths=[out["wavelengths"][q, :n[q]].copy() for q in range(Q)],
                all_flux=[out["flux"][q, :n[q]].copy() for q in range(Q)],
                all_noise_variance=[out["noise_variance"][q, :n[q]].copy() for q in range(Q)],
                all_pixel_mask=[out["pixel_mask"][q, :n[q]].astype(bool) for q in range(Q)],
                all_normalizers=out["normalizers"], filter_flags=out["filter_flags"])


def preload_qsos_device(flux, loglam, ivar, and_mask, lengths, z_qsos, filter_flags=None, params: Parameters = DEFAULT,
                        L_out: int = 1280, stream: int = 0):
    """Device-resident form: torch CUDA tensors in ([Q x L_in] planes), padded [Q x L_out] planes + lengths out --
    exactly the arguments of ``DLAProcessor.process_device`` -- so real spectra never return to the host."""
    import torch
    lib = _lib.load()
    Q, L_in = flux.shape
    dev = flux.device
    out = dict(wavelengths=torch.empty((Q, L_out), dtype=torch.float64, device=dev),
               flux=torch.empty((Q, L_out), dtype=torch.float64, device=dev),
               noise_variance=torch.empty((Q, L_out), dtype=torch.float64, device=dev),
               pixel_mask=torch.empty((Q, L_out), dtype=torch.uint8, device=dev),
               lengths=torch.empty(Q, dtype=torch.int32, device=dev),
               normalizers=torch.empty(Q, dtype=torch.float64, device=dev),
               filter_flags=torch.empty(Q, dtype=torch.uint8, device=dev))
    p = _lib.GpdlaPreloadParams()
    lib.gpdla_default_preload_parameters(ctypes.byref(p))
    p.min_lambda, p.max_lambda = params.min_lambda, params.max_lambda
    p.loading_min_lambda, p.loading_max_lambda = params.loading_min_lambda, params.loading_max_lambda
    p.min_num_pixels = params.min_num_pixels
    ptr = lambda t: None if t is None else ctypes.c_void_p(t.data_ptr())
    with torch.cuda.device(dev):
        _lib.check(lib.gpdla_preload_qsos_device(Q, L_in, ptr(flux), ptr(loglam), ptr(ivar), ptr(and_mask), ptr(lengths),
                                                 ptr(z_qsos), ptr(filter_flags), ctypes.byref(p), L_out,
                                                 ptr(out["wavelengths"]), ptr(out["flux"]), ptr(out["noise_variance"]),
                                                 ptr(out["pixel_mask"]), ptr(out["lengths"]), ptr(out["normalizers"]),
                                                 ptr(out["filter_flags"]), ctypes.c_void_p(stream)))
    return out


def _forest_arrays(num_forest_lines, all_transition_wavelengths, all_oscillator_strengths):
    nl = int(num_forest_lines)
    if nl == 0:
        return 0, None, None
    tw, osc = _f64(all_transition_wavelengths).ravel(), _f64(all_oscillator_strengths).ravel()
    if not (1 <= nl <= _lib.MAX_LINES) or tw.size < nl or osc.size < nl:
        raise ValueError("num_forest_lines must be 1..31 with that many transition wavelengths and oscillator strengths")
    return nl, tw, osc


def objective_lyseries(x, centered_rest_fluxes, lya_1pzs, rest_noise_variances, num_forest_lines,
                       all_transition_wavelengths, all_oscillator_strengths, device: int = 0):
    """``[f, g] = objective_lyseries(x, centered_rest_fluxes, lya_1pzs, rest_noise_variances, num_forest_lines,
    all_transition_wavelengths, all_oscillator_strengths)`` of multi_dlas/objective_lyseries.m:13-87 on the GPU: the
    training objective with the Lyman-series effective optical depth (multi_dlas/spectrum_loss_lyseries.m:20-47).
    ``num_forest_lines = 0`` is ``objective``."""
    import torch
    lib = _lib.load()
    y, z1, nv, xx = _f64(centered_rest_fluxes), _f64(lya_1pzs), _f64(rest_noise_variances), _f64(x)
    N, P = y.shape
    k = (xx.size - 3) // P - 1                                            # objective.m:17
    if xx.size != P * (k + 1) + 3 or z1.shape != y.shape or nv.shape != y.shape:
        raise ValueError("x must have num_pixels * (k + 1) + 3 entries and the three data matrices one shape")
    nl, tw, osc = _forest_arrays(num_forest_lines, all_transition_wavelengths, all_oscillator_strengths)
    f = np.zeros(1); g = np.zeros(xx.size)
    vp = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    with torch.cuda.device(device):
        _lib.check(lib.gpdla_objective_lyseries(N, P, k, vp(y), vp(z1), vp(nv), nl, _dp(tw) if nl else None,
                                                _dp(osc) if nl else None, vp(xx), vp(f), vp(g)))
    return float(f[0]), g


def objective(x, centered_rest_fluxes, lya_1pzs, rest_noise_variances, device: int = 0):
    """``[f, g] = objective(x, centered_rest_fluxes, lya_1pzs, rest_noise_variances)`` of objective.m:12-73 on the
    GPU: negative log-likelihood of the training set and its gradient, ``x = [M(:); log_omega; log c_0; log tau_0;
    log beta]`` (M column-major as in MATLAB).  Host arrays in, ``(float, ndarray)`` out."""
    return objective_lyseries(x, centered_rest_fluxes, lya_1pzs, rest_noise_variances, 0, None, None, device)


class TrainingObjective:
    """The training matrices of learn_qso_model.m:36-75 resident on one GPU; ``ev(x) -> (f, g)`` evaluates
    objective.m for a parameter vector (what minFunc calls at learn_qso_model.m:97-99), uploading only ``x``.
    The matrices are host arrays (uploaded once) or contiguous float64 CUDA tensors on ``device`` (used in place)."""

    def __init__(self, centered_rest_fluxes, lya_1pzs, rest_noise_variances, k: int, device: int = 0,
                 num_forest_lines: int = 0, all_transition_wavelengths=None, all_oscillator_strengths=None):
        """``num_forest_lines > 0`` selects objective_lyseries.m (learn_qso_model_meanflux.m:140-142)."""
        import torch
        self.nl, self.tw, self.osc = _forest_arrays(num_forest_lines, all_transition_wavelengths, all_oscillator_strengths)
        self._lib = _lib.load()
        self._torch = torch
        self.dev = torch.device("cuda", device)
        self.k = int(k)
        cuda_in = [torch.is_tensor(a) and a.is_cuda for a in (centered_rest_fluxes, lya_1pzs, rest_noise_variances)]
        if any(cuda_in):
            # device-resident matrices (e.g. from training_set_device) are kept as they are, without a copy
            mats = (centered_rest_fluxes, lya_1pzs, rest_noise_variances)
            if not all(cuda_in) or any(a.dtype != torch.float64 or not a.is_contiguous() or a.device != self.dev
                                       or a.dim() != 2 or a.shape != mats[0].shape for a in mats):
                raise ValueError("CUDA training matrices must be three contiguous float64 tensors of one (N, P) shape "
                                 "on %s" % self.dev)
            self.N, self.P = tuple(centered_rest_fluxes.shape)
            self.y, self.z1, self.nv = mats
        else:
            self.N, self.P = np.shape(centered_rest_fluxes)
            up = lambda a: torch.from_numpy(_f64(a)).to(self.dev)
            self.y, self.z1, self.nv = up(centered_rest_fluxes), up(lya_1pzs), up(rest_noise_variances)
        self.nx = self.P * (self.k + 1) + 3
        self.x = torch.empty(self.nx, dtype=torch.float64, device=self.dev)
        self.g = torch.empty(self.nx, dtype=torch.float64, device=self.dev)
        self.f = torch.empty(1, dtype=torch.float64, device=self.dev)

    def evaluate_device(self, x_dev, stream: int = 0):
        """x on the device -> (f, g) device tensors (asynchronous)."""
        ptr = lambda t: ctypes.c_void_p(t.data_ptr())
        with self._torch.cuda.device(self.dev):
            _lib.check(self._lib.gpdla_objective_lyseries_device(
                self.N, self.P, self.k, ptr(self.y), ptr(self.z1), ptr(self.nv), self.nl, _dp(self.tw) if self.nl else None,
                _dp(self.osc) if self.nl else None, ptr(x_dev), ptr(self.f), ptr(self.g), ctypes.c_void_p(stream)))
        return self.f, self.g

    def __call__(self, x):
        xx = _f64(x)
        if xx.size != self.nx:
            raise ValueError("x must have %d entries" % self.nx)
        self.x.copy_(self._torch.from_numpy(xx))
        f, g = self.evaluate_device(self.x)
        return float(f.item()), g.cpu().numpy()

    def close(self):
        self.y = self.z1 = self.nv = self.x = self.g = self.f = None


def learn_qso_model(centered_rest_fluxes, lya_1pzs, rest_noise_variances, initial_x, k: int, max_iter: int = 2000,
                    device: int = 0, num_forest_lines: int = 0, all_transition_wavelengths=None,
                    all_oscillator_strengths=None):
    """The optimisation of learn_qso_model.m:97-99 (minFunc L-BFGS there, SciPy's L-BFGS-B here) with the objective and
    gradient evaluated on the GPU.  Returns ``(x, f, scipy_result)``; M = x[:P k].reshape(k, P).T etc. (:101-110).
    ``num_forest_lines > 0`` with the two Lyman-series tables fits objective_lyseries.m instead
    (learn_qso_model_meanflux.m:140-142)."""
    from scipy.optimize import minimize
    ev = TrainingObjective(centered_rest_fluxes, lya_1pzs, rest_noise_variances, k, device, num_forest_lines,
                           all_transition_wavelengths, all_oscillator_strengths)
    try:
        res = minimize(lambda v: ev(v), _f64(initial_x), jac=True, method="L-BFGS-B", options={"maxiter": max_iter})
    finally:
        ev.close()
    return res.x, float(res.fun), res


# ---------------------------------------------------------------- training set + PCA initialisation
def rest_wavelengths(params: Parameters = DEFAULT) -> np.ndarray:
    """The model grid min_lambda:dlambda:max_lambda (learn_qso_model.m:29): 911.75:0.25:1215.75, 1217 exact values."""
    n = int(round((params.max_lambda - params.min_lambda) / params.dlambda)) + 1
    return params.min_lambda + params.dlambda * np.arange(n)


def _check_observed(num_observed: np.ndarray, rest: np.ndarray):
    """nanmean / nanstd of a rest pixel need two observations (learn_qso_model.m:71-95)."""
    few = np.flatnonzero(num_observed < 2)
    if few.size:
        p = int(few[0])
        raise ValueError("rest wavelength %.2f A is observed in %d training spectra; every rest pixel needs at least 2 "
                         "(%d pixels fall short)" % (rest[p], int(num_observed[p]), few.size))


def _initial_x(cov: np.ndarray, std_dev: np.ndarray, k: int, rest: np.ndarray, params: Parameters) -> np.ndarray:
    """learn_qso_model.m:82-95: the top-k principal axes of the pairwise covariance scaled by sqrt(latent), pca's sign
    convention (largest |entry| of each axis positive, first on ties), then log nanstd and the initial c_0, tau_0, beta:
    ``initial_x = [initial_M(:); initial_log_omega; log c_0; log tau_0; log beta]``.  The P x P eigendecomposition runs
    on the host (numpy eigh)."""
    P = cov.shape[0]
    if not 1 <= k < P:
        raise ValueError("k must lie in [1, %d)" % P)
    bad = np.argwhere(np.isnan(cov))
    if bad.size:
        p, q = bad[0]
        raise ValueError("pairwise covariance is undefined at rest wavelengths %.2f / %.2f A: fewer than 2 training "
                         "spectra observe both" % (rest[p], rest[q]))
    latent, coeff = np.linalg.eigh(cov)
    order = np.arange(P)[::-1][:k]                                     # descending
    latent, coeff = latent[order], coeff[:, order]
    if np.any(latent <= 0):
        raise ValueError("the top %d eigenvalues of the pairwise covariance must be positive (smallest: %.3e)"
                         % (k, latent.min()))
    big = np.argmax(np.abs(coeff), axis=0)
    coeff = coeff * np.where(coeff[big, np.arange(k)] < 0, -1.0, 1.0)
    initial_M = coeff * np.sqrt(latent)
    return np.concatenate([initial_M.T.ravel(), np.log(std_dev),
                           [np.log(params.initial_c_0), np.log(params.initial_tau_0), np.log(params.initial_beta)]])


def pairwise_covariance(X, device: int = 0):
    """The covariance ``pca(X, 'rows', 'pairwise')`` decomposes (learn_qso_model.m:82-95) on the GPU: ``X`` [N x P]
    with NaN = not observed -> ``(cov, counts)``, [P x P] each; ``cov`` is NaN where fewer than 2 rows observe a pair."""
    import torch
    lib = _lib.load()
    X = _f64(X)
    if X.ndim != 2:
        raise ValueError("X must be a 2-D (N, P) array")
    N, P = X.shape
    cov, counts = np.empty((P, P)), np.empty((P, P), dtype=np.int32)
    vp = lambda a: ctypes.c_void_p(a.ctypes.data)
    with torch.cuda.device(device):
        _lib.check(lib.gpdla_pairwise_covariance(N, P, vp(X), vp(cov), vp(counts)))
    return cov, counts


def training_set(spectra: Dict, k: int, params: Parameters = DEFAULT, device: int = 0) -> Dict[str, np.ndarray]:
    """The training matrices of learn_qso_model.m:36-75 and the PCA starting point of :82-95 on the GPU, host arrays in
    and out.  ``spectra``: the ragged lists of ``preload_qsos`` or the padded planes (``wavelengths``, ``flux``,
    ``noise_variance``, ``pixel_mask``, ``lengths``), plus ``z_qsos``, for the training selection.  Returns
    ``rest_wavelengths``, ``lya_1pzs``, ``centered_rest_fluxes``, ``rest_noise_variances`` ([N x P]), ``mu``,
    ``std_dev``, ``num_observed`` ([P]) and ``initial_x`` -- the arguments of ``learn_qso_model``."""
    import torch
    lib = _lib.load()
    sp = pad_spectra(spectra)
    W, F, V = _f64(sp["wavelengths"]), _f64(sp["flux"]), _f64(sp["noise_variance"])
    Mk = np.ascontiguousarray(sp["pixel_mask"], dtype=np.uint8)
    lengths = np.ascontiguousarray(sp["lengths"], dtype=np.int32).ravel()
    z = _f64(sp["z_qsos"]).ravel()
    _check_planes(W, F, V, Mk, lengths, z)
    N, L_max = W.shape
    rest = rest_wavelengths(params)
    P = rest.size
    out = dict(rest_wavelengths=rest, lya_1pzs=np.empty((N, P)), centered_rest_fluxes=np.empty((N, P)),
               rest_noise_variances=np.empty((N, P)), mu=np.empty(P), std_dev=np.empty(P),
               num_observed=np.full(P, np.iinfo(np.int32).max, dtype=np.int32))
    vp = lambda a: ctypes.c_void_p(a.ctypes.data)
    cov, counts = np.empty((P, P)), np.empty((P, P), dtype=np.int32)
    with torch.cuda.device(device):
        rc = lib.gpdla_training_set(N, L_max, vp(W), vp(F), vp(V), vp(Mk), vp(lengths), vp(z), vp(rest), P,
                                    lya_wavelength, float(params.max_noise_variance), vp(out["lya_1pzs"]),
                                    vp(out["centered_rest_fluxes"]), vp(out["rest_noise_variances"]), vp(out["mu"]),
                                    vp(out["std_dev"]), vp(out["num_observed"]))
        if rc == _lib.GPDLA_ERR_INVALID:
            _check_observed(out["num_observed"], rest)
        _lib.check(rc)
        _lib.check(lib.gpdla_pairwise_covariance(N, P, vp(out["centered_rest_fluxes"]), vp(cov), vp(counts)))
    out["initial_x"] = _initial_x(cov, out["std_dev"], int(k), rest, params)
    return out


def training_set_device(wavelengths, flux, noise_variance, pixel_mask, lengths, z_qsos, k: int,
                        params: Parameters = DEFAULT) -> Dict:
    """Device-resident ``training_set``: the CUDA tensors ``preload_qsos_device`` returns (float64 [N x L_max] planes,
    uint8 mask, int32 lengths -- a negative or zero length gives an all-NaN row -- and float64 ``z_qsos``) in, the same
    names as CUDA tensors out (``initial_x`` on the host).  Only the [P x P] covariance, ``std_dev`` and
    ``num_observed`` cross to the host, for the eigendecomposition."""
    import torch
    lib = _lib.load()
    dev = wavelengths.device
    N, L_max = wavelengths.shape
    for t, dt in ((wavelengths, torch.float64), (flux, torch.float64), (noise_variance, torch.float64),
                  (pixel_mask, torch.uint8), (lengths, torch.int32), (z_qsos, torch.float64)):
        if not (t.is_cuda and t.device == dev and t.dtype == dt and t.is_contiguous()):
            raise ValueError("training_set_device takes contiguous CUDA tensors on one device: float64 planes, uint8 "
                             "pixel_mask, int32 lengths, float64 z_qsos")
    if any(t.shape != wavelengths.shape for t in (flux, noise_variance, pixel_mask)) or \
            lengths.shape != (N,) or z_qsos.shape != (N,):
        raise ValueError("wavelengths, flux, noise_variance and pixel_mask must share one (N, L_max) shape and lengths, "
                         "z_qsos have one entry per spectrum")
    rest = rest_wavelengths(params)
    P = rest.size
    f64 = dict(dtype=torch.float64, device=dev)
    out = dict(rest_wavelengths=torch.from_numpy(rest).to(dev), lya_1pzs=torch.empty((N, P), **f64),
               centered_rest_fluxes=torch.empty((N, P), **f64), rest_noise_variances=torch.empty((N, P), **f64),
               mu=torch.empty(P, **f64), std_dev=torch.empty(P, **f64),
               num_observed=torch.empty(P, dtype=torch.int32, device=dev))
    cov = torch.empty((P, P), **f64)
    counts = torch.empty((P, P), dtype=torch.int32, device=dev)
    ptr = lambda t: ctypes.c_void_p(t.data_ptr())
    with torch.cuda.device(dev):
        stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        _lib.check(lib.gpdla_training_set_device(
            N, L_max, ptr(wavelengths), ptr(flux), ptr(noise_variance), ptr(pixel_mask), ptr(lengths), ptr(z_qsos),
            ptr(out["rest_wavelengths"]), P, lya_wavelength, float(params.max_noise_variance), ptr(out["lya_1pzs"]),
            ptr(out["centered_rest_fluxes"]), ptr(out["rest_noise_variances"]), ptr(out["mu"]), ptr(out["std_dev"]),
            ptr(out["num_observed"]), stream))
        _lib.check(lib.gpdla_pairwise_covariance_device(N, P, ptr(out["centered_rest_fluxes"]), ptr(cov), ptr(counts),
                                                        stream))
        num_observed = out["num_observed"].cpu().numpy()
        _check_observed(num_observed, rest)
        out["initial_x"] = _initial_x(cov.cpu().numpy(), out["std_dev"].cpu().numpy(), int(k), rest, params)
    return out


def learn_qso_model_from_spectra(spectra: Dict, k: int, params: Parameters = DEFAULT, max_iter: int = 2000,
                                 device: int = 0) -> Dict:
    """learn_qso_model.m:36-110 from preprocessed training spectra (ragged or padded, plus ``z_qsos``): the training
    set and PCA starting point (``training_set_device``), L-BFGS on the GPU objective (``learn_qso_model``) and the
    unpacking of :101-110.  Returns the model ``DLAProcessor`` takes -- ``rest_wavelengths``, ``mu``, ``M`` (P x k),
    ``log_omega``, ``log_c_0``, ``log_tau_0``, ``log_beta`` -- plus ``initial_x``, ``log_likelihood`` (the objective
    value at the optimum, the negative log-likelihood that learn_qso_model.m stores under this name) and the SciPy
    ``result``."""
    import torch
    sp = pad_spectra(spectra)
    W, F, V = _f64(sp["wavelengths"]), _f64(sp["flux"]), _f64(sp["noise_variance"])
    Mk = np.ascontiguousarray(sp["pixel_mask"], dtype=np.uint8)
    lengths = np.ascontiguousarray(sp["lengths"], dtype=np.int32).ravel()
    z = _f64(sp["z_qsos"]).ravel()
    _check_planes(W, F, V, Mk, lengths, z)
    dev = torch.device("cuda", device)
    up = lambda a: torch.from_numpy(a).to(dev)
    ts = training_set_device(up(W), up(F), up(V), up(Mk), up(lengths), up(z), k, params)
    x, f, res = learn_qso_model(ts["centered_rest_fluxes"], ts["lya_1pzs"], ts["rest_noise_variances"],
                                ts["initial_x"], k, max_iter, device)
    P = ts["mu"].numel()
    return dict(rest_wavelengths=ts["rest_wavelengths"].cpu().numpy(), mu=ts["mu"].cpu().numpy(),
                M=np.ascontiguousarray(x[:P * k].reshape(k, P).T), log_omega=x[P * k:P * (k + 1)].copy(),
                log_c_0=float(x[-3]), log_tau_0=float(x[-2]), log_beta=float(x[-1]),
                initial_x=ts["initial_x"], log_likelihood=f, result=res)


# ---------------------------------------------------------------- the multi-DLA (mean-flux) model's training set
def _check_forest_lines(num_forest_lines) -> int:
    nl = int(num_forest_lines)
    if not 0 <= nl <= _lib.MAX_LINES:
        raise ValueError("num_forest_lines must lie in [0, %d]" % _lib.MAX_LINES)
    return nl


def row_nanmedian_fill(X, device: int = 0) -> np.ndarray:
    """A copy of ``X`` [N x P] with each row's NaNs replaced by that row's nanmedian (MATLAB's median, ``meanof`` for an
    even count) on the GPU; an all-NaN row stays NaN.  The matrix learn_qso_model_meanflux.m decomposes with
    ``pca(..., 'rows', 'complete')``."""
    import torch
    lib = _lib.load()
    X = _f64(X)
    if X.ndim != 2:
        raise ValueError("X must be a 2-D (N, P) array")
    N, P = X.shape
    out = np.empty((N, P))
    with torch.cuda.device(device):
        _lib.check(lib.gpdla_row_nanmedian_fill(N, P, ctypes.c_void_p(X.ctypes.data), ctypes.c_void_p(out.ctypes.data)))
    return out


def training_set_meanflux(spectra: Dict, k: int, params: Parameters = MULTI, num_forest_lines: int = 31,
                          device: int = 0) -> Dict[str, np.ndarray]:
    """The training matrices and PCA starting point of multi_dlas/learn_qso_model_meanflux.m on the GPU, host arrays in
    and out: ``training_set`` with the Lyman-series mean-flux suppression (Kim et al. 2007, fixed prev_tau_0 = 0.0023,
    prev_beta = 3.65, the first ``num_forest_lines`` members) divided out of the rest fluxes and noise variances, the
    noise ceiling ``params.max_noise_variance`` (``MULTI``: 3^2), and the PCA of the row-nanmedian-filled centred fluxes
    (``pca(..., 'rows', 'complete')``).  Returns the names ``training_set`` returns plus ``lya_absorption`` [N x P]."""
    import torch
    lib = _lib.load()
    nl = _check_forest_lines(num_forest_lines)
    sp = pad_spectra(spectra)
    W, F, V = _f64(sp["wavelengths"]), _f64(sp["flux"]), _f64(sp["noise_variance"])
    Mk = np.ascontiguousarray(sp["pixel_mask"], dtype=np.uint8)
    lengths = np.ascontiguousarray(sp["lengths"], dtype=np.int32).ravel()
    z = _f64(sp["z_qsos"]).ravel()
    _check_planes(W, F, V, Mk, lengths, z)
    N, L_max = W.shape
    rest = rest_wavelengths(params)
    P = rest.size
    out = dict(rest_wavelengths=rest, lya_1pzs=np.empty((N, P)), centered_rest_fluxes=np.empty((N, P)),
               rest_noise_variances=np.empty((N, P)), lya_absorption=np.empty((N, P)), mu=np.empty(P),
               std_dev=np.empty(P), num_observed=np.full(P, np.iinfo(np.int32).max, dtype=np.int32))
    vp = lambda a: ctypes.c_void_p(a.ctypes.data)
    filled = np.empty((N, P))
    cov, counts = np.empty((P, P)), np.empty((P, P), dtype=np.int32)
    with torch.cuda.device(device):
        rc = lib.gpdla_training_set_lyseries(N, L_max, vp(W), vp(F), vp(V), vp(Mk), vp(lengths), vp(z), vp(rest), P,
                                             lya_wavelength, float(params.max_noise_variance), nl, vp(out["lya_1pzs"]),
                                             vp(out["centered_rest_fluxes"]), vp(out["rest_noise_variances"]),
                                             vp(out["lya_absorption"]), vp(out["mu"]), vp(out["std_dev"]),
                                             vp(out["num_observed"]))
        if rc == _lib.GPDLA_ERR_INVALID:
            _check_observed(out["num_observed"], rest)
        _lib.check(rc)
        _lib.check(lib.gpdla_row_nanmedian_fill(N, P, vp(out["centered_rest_fluxes"]), vp(filled)))
        _lib.check(lib.gpdla_pairwise_covariance(N, P, vp(filled), vp(cov), vp(counts)))
    out["initial_x"] = _initial_x(cov, out["std_dev"], int(k), rest, params)
    return out


def training_set_meanflux_device(wavelengths, flux, noise_variance, pixel_mask, lengths, z_qsos, k: int,
                                 params: Parameters = MULTI, num_forest_lines: int = 31) -> Dict:
    """Device-resident ``training_set_meanflux``: the CUDA tensors ``preload_qsos_device`` returns in, the same names as
    CUDA tensors out (``initial_x`` on the host).  The filled copy lives only for the covariance; only the [P x P]
    covariance, ``std_dev`` and ``num_observed`` cross to the host."""
    import torch
    lib = _lib.load()
    nl = _check_forest_lines(num_forest_lines)
    dev = wavelengths.device
    N, L_max = wavelengths.shape
    for t, dt in ((wavelengths, torch.float64), (flux, torch.float64), (noise_variance, torch.float64),
                  (pixel_mask, torch.uint8), (lengths, torch.int32), (z_qsos, torch.float64)):
        if not (t.is_cuda and t.device == dev and t.dtype == dt and t.is_contiguous()):
            raise ValueError("training_set_meanflux_device takes contiguous CUDA tensors on one device: float64 planes, "
                             "uint8 pixel_mask, int32 lengths, float64 z_qsos")
    if any(t.shape != wavelengths.shape for t in (flux, noise_variance, pixel_mask)) or \
            lengths.shape != (N,) or z_qsos.shape != (N,):
        raise ValueError("wavelengths, flux, noise_variance and pixel_mask must share one (N, L_max) shape and lengths, "
                         "z_qsos have one entry per spectrum")
    rest = rest_wavelengths(params)
    P = rest.size
    f64 = dict(dtype=torch.float64, device=dev)
    out = dict(rest_wavelengths=torch.from_numpy(rest).to(dev), lya_1pzs=torch.empty((N, P), **f64),
               centered_rest_fluxes=torch.empty((N, P), **f64), rest_noise_variances=torch.empty((N, P), **f64),
               lya_absorption=torch.empty((N, P), **f64), mu=torch.empty(P, **f64), std_dev=torch.empty(P, **f64),
               num_observed=torch.empty(P, dtype=torch.int32, device=dev))
    filled = torch.empty((N, P), **f64)
    cov = torch.empty((P, P), **f64)
    counts = torch.empty((P, P), dtype=torch.int32, device=dev)
    ptr = lambda t: ctypes.c_void_p(t.data_ptr())
    with torch.cuda.device(dev):
        stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        _lib.check(lib.gpdla_training_set_lyseries_device(
            N, L_max, ptr(wavelengths), ptr(flux), ptr(noise_variance), ptr(pixel_mask), ptr(lengths), ptr(z_qsos),
            ptr(out["rest_wavelengths"]), P, lya_wavelength, float(params.max_noise_variance), nl, ptr(out["lya_1pzs"]),
            ptr(out["centered_rest_fluxes"]), ptr(out["rest_noise_variances"]), ptr(out["lya_absorption"]),
            ptr(out["mu"]), ptr(out["std_dev"]), ptr(out["num_observed"]), stream))
        _lib.check(lib.gpdla_row_nanmedian_fill_device(N, P, ptr(out["centered_rest_fluxes"]), ptr(filled), stream))
        _lib.check(lib.gpdla_pairwise_covariance_device(N, P, ptr(filled), ptr(cov), ptr(counts), stream))
        num_observed = out["num_observed"].cpu().numpy()
        _check_observed(num_observed, rest)
        out["initial_x"] = _initial_x(cov.cpu().numpy(), out["std_dev"].cpu().numpy(), int(k), rest, params)
    return out


def learn_qso_model_meanflux_from_spectra(spectra: Dict, k: int, params: Parameters = MULTI, max_iter: int = 2000,
                                          device: int = 0) -> Dict:
    """multi_dlas/learn_qso_model_meanflux.m from preprocessed training spectra (ragged or padded, plus ``z_qsos``): the
    mean-flux training set and its PCA starting point (``training_set_meanflux_device``), L-BFGS on the GPU
    objective_lyseries with 31 Lyman-series members, and the unpacking of learn_qso_model.m:101-110.  Returns the model
    ``process_qsos_multiple_dlas_meanflux`` / ``DLAProcessor.process_multi`` load plus ``initial_x``,
    ``log_likelihood`` and the SciPy ``result``, as ``learn_qso_model_from_spectra`` does."""
    import torch
    sp = pad_spectra(spectra)
    W, F, V = _f64(sp["wavelengths"]), _f64(sp["flux"]), _f64(sp["noise_variance"])
    Mk = np.ascontiguousarray(sp["pixel_mask"], dtype=np.uint8)
    lengths = np.ascontiguousarray(sp["lengths"], dtype=np.int32).ravel()
    z = _f64(sp["z_qsos"]).ravel()
    _check_planes(W, F, V, Mk, lengths, z)
    dev = torch.device("cuda", device)
    up = lambda a: torch.from_numpy(a).to(dev)
    nl = _params.num_forest_lines
    ts = training_set_meanflux_device(up(W), up(F), up(V), up(Mk), up(lengths), up(z), k, params, nl)
    x, f, res = learn_qso_model(ts["centered_rest_fluxes"], ts["lya_1pzs"], ts["rest_noise_variances"],
                                ts["initial_x"], k, max_iter, device, nl, _params.all_transition_wavelengths,
                                _params.all_oscillator_strengths)
    P = ts["mu"].numel()
    return dict(rest_wavelengths=ts["rest_wavelengths"].cpu().numpy(), mu=ts["mu"].cpu().numpy(),
                M=np.ascontiguousarray(x[:P * k].reshape(k, P).T), log_omega=x[P * k:P * (k + 1)].copy(),
                log_c_0=float(x[-3]), log_tau_0=float(x[-2]), log_beta=float(x[-1]),
                initial_x=ts["initial_x"], log_likelihood=f, result=res)


# ---------------------------------------------------------------- population statistics (CDDF_analysis/calc_cddf.py)
def dla_statistics_width(n_z: int, n_nhi: int) -> int:
    """Length of the sums vector for n_z z bins and n_nhi log-N bins."""
    return 2 * n_z * n_nhi + 5 * n_z + 1


def dla_statistics_layout(n_z: int, n_nhi: int) -> Dict[str, tuple]:
    """Names of the parts of the sums vector -> (start, shape): counts, counts_var [n_z, n_nhi]; dla, dla_var, nhi,
    nhi_var, path [n_z]; num_quasars []."""
    a, t = n_z * n_nhi, 2 * n_z * n_nhi
    return dict(counts=(0, (n_z, n_nhi)), counts_var=(a, (n_z, n_nhi)), dla=(t, (n_z,)), dla_var=(t + n_z, (n_z,)),
                nhi=(t + 2 * n_z, (n_z,)), nhi_var=(t + 3 * n_z, (n_z,)), path=(t + 4 * n_z, (n_z,)),
                num_quasars=(t + 5 * n_z, ()))


def unpack_dla_statistics(sums, n_z: int, n_nhi: int) -> Dict[str, np.ndarray]:
    """The sums vector (host array or tensor) -> a dict of its parts as host arrays."""
    v = np.asarray(sums.cpu().numpy() if hasattr(sums, "cpu") else sums, dtype=np.float64)
    out = {}
    for n, (start, shape) in dla_statistics_layout(n_z, n_nhi).items():
        size = int(np.prod(shape))
        out[n] = v[start:start + size].reshape(shape).copy() if shape else float(v[start])
    return out


def _stats_edges(z_edges, log_nhi_edges):
    ze, ne = _f64(z_edges).ravel(), _f64(log_nhi_edges).ravel()
    if ze.size < 2 or ne.size < 2:
        raise ValueError("z_edges and log_nhi_edges need at least two entries (one bin)")
    return ze, ne


def dla_statistics_sums(results: Dict, samples: Dict, z_edges, log_nhi_edges, select=None, sums=None,
                        dla_log_nhi_min: float = _params.dla_log_nhi_min, omega_m: float = _params.omega_m,
                        device: int = 0) -> np.ndarray:
    """The additive sums behind the column density distribution, dN/dX and Omega_DLA (CDDF_analysis/calc_cddf.py) of
    one ``process`` / ``process_qsos`` result (host arrays, with ``sample_log_likelihoods_dla``) and the samples it was
    run with, computed on the GPU.  Per quasar the normalised sample posterior is binned by z_dla (``z_edges``) and
    log10 N_HI (``log_nhi_edges``), half-open bins; ``select`` [Q] (bool) drops quasars (SNR, z_qso or filter cuts).
    Returns the float64 vector ``dla_statistics_layout`` describes -- ``sums`` (when given) plus this batch.  Sums of
    disjoint quasar sets add; pass the total to ``finish_dla_statistics``.  Variances add across quasars, not across z
    bins: a statistic over all z needs a single z bin."""
    import torch
    lib = _lib.load()
    ze, ne = _stats_edges(z_edges, log_nhi_edges)
    width = dla_statistics_width(ze.size - 1, ne.size - 1)
    ll = _f64(results["sample_log_likelihoods_dla"])
    if ll.ndim != 2:
        raise ValueError("sample_log_likelihoods_dla must be (Q, S)")
    Q, S = ll.shape
    p, zlo, zhi = (_f64(results[n]).ravel() for n in ("p_dlas", "min_z_dlas", "max_z_dlas"))
    off, lnhi, nhi = (_f64(samples[k]).ravel() for k in ("offset_samples", "log_nhi_samples", "nhi_samples"))
    if p.size != Q or zlo.size != Q or zhi.size != Q or off.size != S or lnhi.size != S or nhi.size != S:
        raise ValueError("results need Q entries per quasar and the samples S entries each (Q, S = %d, %d)" % (Q, S))
    sel = None
    if select is not None:
        sel = np.ascontiguousarray(np.asarray(select).astype(np.uint8)).ravel()
        if sel.size != Q:
            raise ValueError("select must have one entry per quasar")
    out = np.zeros(width) if sums is None else _f64(sums).ravel().copy()
    if out.size != width:
        raise ValueError("sums must have %d entries" % width)
    vp = lambda a: None if a is None else ctypes.c_void_p(a.ctypes.data)
    with torch.cuda.device(device):
        _lib.check(lib.gpdla_dla_statistics(Q, S, vp(ll), vp(p), vp(zlo), vp(zhi), vp(sel), vp(off), vp(lnhi), vp(nhi),
                                            ze.size - 1, _dp(ze), ne.size - 1, _dp(ne), float(dla_log_nhi_min),
                                            float(omega_m), vp(out)))
    return out


def multi_dla_statistics_sums(results: Dict, samples: Dict, z_edges, log_nhi_edges, select=None, sums=None,
                              dla_log_nhi_min: float = _params.dla_log_nhi_min, omega_m: float = _params.omega_m,
                              device: int = 0) -> np.ndarray:
    """``dla_statistics_sums`` for the multi-DLA model (Ho et al. 2021), computed on the GPU, from one
    ``process_multi`` / ``process_qsos_multiple_dlas_meanflux`` result in the reference layout --
    ``sample_log_likelihoods_dla`` (Q, S, J), ``base_sample_inds`` (Q, S, J-1), 0-based, ``model_posteriors``
    (Q, 2 + J) -- and the samples it was run with.  Each quasar adds the exact mean and variance, under its model
    mixture, of the number of absorbers per cell (and of the N_HI sum per z bin); a j-DLA sample places j absorbers,
    the sub-DLA model none.  Same layout, ``select``, ``sums`` and finishing as ``dla_statistics_sums``."""
    import torch
    lib = _lib.load()
    ze, ne = _stats_edges(z_edges, log_nhi_edges)
    width = dla_statistics_width(ze.size - 1, ne.size - 1)
    sll = np.asarray(results["sample_log_likelihoods_dla"], dtype=np.float64)
    if sll.ndim != 3:
        raise ValueError("sample_log_likelihoods_dla must be (Q, S, max_dlas)")
    Q, S, J = sll.shape
    ll = np.ascontiguousarray(np.transpose(sll, (0, 2, 1)))
    part = None
    if J > 1:
        bsi = np.asarray(results["base_sample_inds"])
        if bsi.shape != (Q, S, J - 1):
            raise ValueError("base_sample_inds must be (Q, S, max_dlas - 1)")
        part = np.ascontiguousarray(np.transpose(bsi, (0, 2, 1)), dtype=np.int32)
    mp = _f64(results["model_posteriors"])
    zlo, zhi = (_f64(results[n]).ravel() for n in ("min_z_dlas", "max_z_dlas"))
    off, lnhi, nhi = (_f64(samples[k]).ravel() for k in ("offset_samples", "log_nhi_samples", "nhi_samples"))
    if mp.shape != (Q, J + 2) or zlo.size != Q or zhi.size != Q or off.size != S or lnhi.size != S or nhi.size != S:
        raise ValueError("results need Q entries per quasar and the samples S entries each (Q, S = %d, %d)" % (Q, S))
    sel = None
    if select is not None:
        sel = np.ascontiguousarray(np.asarray(select).astype(np.uint8)).ravel()
        if sel.size != Q:
            raise ValueError("select must have one entry per quasar")
    out = np.zeros(width) if sums is None else _f64(sums).ravel().copy()
    if out.size != width:
        raise ValueError("sums must have %d entries" % width)
    vp = lambda a: None if a is None else ctypes.c_void_p(a.ctypes.data)
    with torch.cuda.device(device):
        _lib.check(lib.gpdla_multi_dla_statistics(Q, S, J, vp(ll), vp(part), vp(mp), vp(zlo), vp(zhi), vp(sel), vp(off),
                                                  vp(lnhi), vp(nhi), ze.size - 1, _dp(ze), ne.size - 1, _dp(ne),
                                                  float(dla_log_nhi_min), float(omega_m), vp(out)))
    return out

def omega_dla_coefficient(hubble_h: float = _params.hubble_h) -> float:
    """8 pi G m_H / (3 c H0) in cm^2: Omega_DLA = this x (sum of N_HI) / (absorption path).  HI only, no helium."""
    H0 = 100.0 * hubble_h * 1e5 / _params.megaparsec                      # s^-1
    return 8.0 * np.pi * _params.gravitational_constant * _params.hydrogen_mass / (3.0 * _params.speed_of_light_cgs * H0)


def finish_dla_statistics(sums, z_edges, log_nhi_edges, hubble_h: float = _params.hubble_h) -> Dict[str, np.ndarray]:
    """The statistics from the total sums (host): ``cddf`` f(N, X) = counts / (dN path) [n_z, n_nhi] in cm^2 per unit
    absorption distance, ``dndx`` = dla / path and ``omega_dla`` = 8 pi G m_H / (3 c H0) nhi / path [n_z], each with
    ``*_sigma`` = sqrt(variance) over the same factors, plus ``path_length`` (sum of dX per z bin), ``expected_counts``
    (the Poisson-binomial mean of DLAs per cell) and ``num_quasars``.  Omega_m entered through the path the sums carry;
    ``hubble_h`` sets H0 = 100 h km/s/Mpc.  Bins without path give NaN."""
    ze, ne = _stats_edges(z_edges, log_nhi_edges)
    n_z, n_nhi = ze.size - 1, ne.size - 1
    t = unpack_dla_statistics(sums, n_z, n_nhi)
    path = t["path"]
    with np.errstate(divide="ignore", invalid="ignore"):
        inv = np.where(path > 0, 1.0 / path, np.nan)
        dn = 10.0 ** ne[1:] - 10.0 ** ne[:-1]
        coef = omega_dla_coefficient(hubble_h)
        return dict(cddf=t["counts"] / dn[None, :] * inv[:, None],
                    cddf_sigma=np.sqrt(t["counts_var"]) / dn[None, :] * inv[:, None],
                    dndx=t["dla"] * inv, dndx_sigma=np.sqrt(t["dla_var"]) * inv,
                    omega_dla=coef * t["nhi"] * inv, omega_dla_sigma=coef * np.sqrt(np.maximum(t["nhi_var"], 0.0)) * inv,
                    path_length=path, expected_counts=t["counts"], num_quasars=int(round(t["num_quasars"])))


def matlab_default_rand(n: int) -> np.ndarray:
    """First ``n`` numbers of MATLAB's ``rng('default'); rand`` stream as the library generates them."""
    out = np.empty(int(n))
    _lib.load().gpdla_matlab_default_rand(_dp(out), int(n))
    return out


def voigt(lambdas: Sequence[float], z: float, N: float, num_lines: int = _lib.MAX_LINES) -> np.ndarray:
    """``profile = voigt(lambdas, z, N [, num_lines])`` (voigt.c:253-304): Voigt absorption profile of the
    first ``num_lines`` Lyman-series members for a cloud of column density ``N`` (cm^-2) at redshift ``z``,
    convolved with the 7-pixel instrument profile; returns ``len(lambdas) - 6`` values."""
    lib = _lib.load()
    lam = _f64(lambdas).ravel()
    out = np.empty(max(lam.size - 6, 0))
    _lib.check(lib.gpdla_voigt(_dp(lam), lam.size, float(z), float(N), int(num_lines), _dp(out)))
    return out


def voigt_batch(lambdas, z, N, num_lines: int = _lib.MAX_LINES):
    """Device-resident batched ``voigt``: CUDA float64 tensors ``lambdas`` (P,), ``z`` (S,), ``N`` (S,) ->
    ``(S, P - 6)`` CUDA tensor, on torch's current stream."""
    import torch
    lib = _lib.load()
    assert lambdas.is_cuda and lambdas.dtype == torch.float64 and z.dtype == torch.float64 and N.dtype == torch.float64
    lambdas, z, N = lambdas.contiguous(), z.contiguous(), N.contiguous()
    out = torch.empty((z.numel(), lambdas.numel() - 6), dtype=torch.float64, device=lambdas.device)
    with torch.cuda.device(lambdas.device):
        stream = torch.cuda.current_stream().cuda_stream
        _lib.check(lib.gpdla_voigt_batch_device(lambdas.data_ptr(), lambdas.numel(), z.data_ptr(), N.data_ptr(),
                                                z.numel(), int(num_lines), out.data_ptr(), ctypes.c_void_p(stream)))
    return out
