"""ctypes binding of libgpdla.so (the C ABI in include/gpdla.h).  Fails loudly when the
library is missing: there is no CPU or PyTorch fallback."""
from __future__ import annotations

import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("GPDLA_LIB", os.path.join(HERE, "libgpdla.so"))   # GPDLA_LIB: debug builds only

c_double_p = ctypes.POINTER(ctypes.c_double)
c_u8_p = ctypes.POINTER(ctypes.c_uint8)
c_i32_p = ctypes.POINTER(ctypes.c_int32)
c_i64_p = ctypes.POINTER(ctypes.c_int64)

GPDLA_OK, GPDLA_ERR_INVALID, GPDLA_ERR_CUDA, GPDLA_ERR_UNSUPPORTED, GPDLA_ERR_STATE = 0, 1, 2, 3, 4
MAX_LINES = 31


class GpdlaParams(ctypes.Structure):
    _fields_ = [("min_lambda", ctypes.c_double), ("max_lambda", ctypes.c_double),
                ("lya_wavelength", ctypes.c_double), ("lyman_limit", ctypes.c_double),
                ("prior_z_qso_increase", ctypes.c_double), ("min_z_cut", ctypes.c_double),
                ("max_z_cut", ctypes.c_double), ("pixel_spacing", ctypes.c_double),
                ("num_lines", ctypes.c_int32), ("batch_quasars", ctypes.c_int32),
                ("gram_digits", ctypes.c_int32), ("rest_table", ctypes.c_int32)]


RESULT_F64 = ["min_z_dlas", "max_z_dlas", "log_priors_no_dla", "log_priors_dla", "log_likelihoods_no_dla",
              "log_likelihoods_dla", "log_posteriors_no_dla", "log_posteriors_dla", "model_posteriors",
              "p_no_dlas", "p_dlas", "sample_log_likelihoods_dla", "map_z_dlas", "map_log_nhis"]


class GpdlaPreloadParams(ctypes.Structure):
    _fields_ = [("loading_min_lambda", ctypes.c_double), ("loading_max_lambda", ctypes.c_double),
                ("normalization_min_lambda", ctypes.c_double), ("normalization_max_lambda", ctypes.c_double),
                ("min_lambda", ctypes.c_double), ("max_lambda", ctypes.c_double),
                ("min_num_pixels", ctypes.c_int32), ("reserved", ctypes.c_int32)]


class GpdlaResults(ctypes.Structure):
    _fields_ = [(n, ctypes.c_void_p) for n in RESULT_F64] + [("map_inds", ctypes.c_void_p)]


MULTI_RESULT_FIELDS = ["min_z_dlas", "max_z_dlas", "log_priors_no_dla", "log_priors_lls", "log_priors_dla",
                       "log_likelihoods_no_dla", "log_likelihoods_lls", "log_likelihoods_dla",
                       "log_posteriors_no_dla", "log_posteriors_lls", "log_posteriors_dla", "model_posteriors",
                       "p_no_dlas", "p_lls", "p_dlas", "MAP_z_dlas", "MAP_log_nhis", "MAP_inds",
                       "sample_log_likelihoods_dla", "sample_log_likelihoods_lls", "base_sample_inds"]


class GpdlaMultiResults(ctypes.Structure):
    _fields_ = [(n, ctypes.c_void_p) for n in MULTI_RESULT_FIELDS]


RECONSTRUCTION_FIELDS = ["absorption", "prior_mean", "prior_sd", "fit_mean", "continuum", "continuum_sd", "latent", "chi2",
                         "log_likelihood", "num_pixels"]


class GpdlaReconstruction(ctypes.Structure):
    _fields_ = [(n, ctypes.c_void_p) for n in RECONSTRUCTION_FIELDS]


class GpdlaDrawOptions(ctypes.Structure):
    _fields_ = [("seed", ctypes.c_uint64), ("first_quasar", ctypes.c_int64), ("model", ctypes.c_int32),
                ("max_dlas", ctypes.c_int32), ("inject", ctypes.c_int32), ("from_prior", ctypes.c_int32),
                ("num_absorbers", ctypes.c_int32), ("reserved", ctypes.c_int32), ("absorber_z", ctypes.c_void_p),
                ("absorber_nhi", ctypes.c_void_p)]


DRAW_FIELDS = ["flux", "absorption", "truth_model", "truth_inds", "truth_z", "truth_log_nhi"]


class GpdlaDrawOutputs(ctypes.Structure):
    _fields_ = [(n, ctypes.c_void_p) for n in DRAW_FIELDS]


# every symbol include/gpdla.h declares: name -> (restype, argtypes)
SYMBOLS = {
    "gpdla_default_parameters": (None, [ctypes.POINTER(GpdlaParams)]),
    "gpdla_create": (ctypes.c_int, [ctypes.POINTER(ctypes.c_void_p), ctypes.c_int]),
    "gpdla_destroy": (None, [ctypes.c_void_p]),
    "gpdla_last_error": (ctypes.c_char_p, [ctypes.c_void_p]),
    "gpdla_launch_count": (ctypes.c_uint64, [ctypes.c_void_p]),
    "gpdla_set_profiling": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int]),
    "gpdla_profile_read": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_double), c_i64_p]),
    "gpdla_set_parameters": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(GpdlaParams)]),
    "gpdla_set_model": (ctypes.c_int, [ctypes.c_void_p, c_double_p, ctypes.c_int32, c_double_p, c_double_p,
                                       ctypes.c_int32, c_double_p, ctypes.c_double, ctypes.c_double,
                                       ctypes.c_double]),
    "gpdla_set_samples": (ctypes.c_int, [ctypes.c_void_p, c_double_p, c_double_p, c_double_p, ctypes.c_int64]),
    "gpdla_set_prior": (ctypes.c_int, [ctypes.c_void_p, c_double_p, c_u8_p, ctypes.c_int64]),
    "gpdla_process_qsos": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64, ctypes.c_void_p,
                                          ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                          ctypes.c_void_p, ctypes.POINTER(GpdlaResults)]),
    "gpdla_process_qsos_device": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64, ctypes.c_void_p,
                                                 ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                                 ctypes.c_void_p, ctypes.c_void_p, ctypes.POINTER(GpdlaResults),
                                                 ctypes.c_void_p]),
    "gpdla_set_lls_samples": (ctypes.c_int, [ctypes.c_void_p, c_double_p, ctypes.c_int64, ctypes.c_double,
                                             ctypes.c_double]),
    "gpdla_process_qsos_multi": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64] + [ctypes.c_void_p] * 6
                                 + [ctypes.c_int32, ctypes.c_void_p, ctypes.POINTER(GpdlaMultiResults)]),
    "gpdla_process_qsos_multi_device": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64]
                                        + [ctypes.c_void_p] * 6 + [ctypes.c_int32, ctypes.c_void_p,
                                                                   ctypes.POINTER(GpdlaMultiResults), ctypes.c_void_p]),
    "gpdla_matlab_default_rand": (None, [c_double_p, ctypes.c_int64]),
    "gpdla_voigt": (ctypes.c_int, [c_double_p, ctypes.c_int64, ctypes.c_double, ctypes.c_double, ctypes.c_int32,
                                   c_double_p]),
    "gpdla_voigt_batch_device": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p,
                                                ctypes.c_int64, ctypes.c_int32, ctypes.c_void_p, ctypes.c_void_p]),
    "gpdla_line_constants": (None, [c_double_p, c_double_p, c_double_p, c_double_p]),
    "gpdla_rest_table": (ctypes.c_int, [ctypes.c_int32, ctypes.c_double, c_double_p, c_i32_p, c_i32_p, c_double_p,
                                        c_double_p]),
    "gpdla_host_alloc": (ctypes.c_int, [ctypes.POINTER(ctypes.c_void_p), ctypes.c_uint64]),
    "gpdla_host_free": (None, [ctypes.c_void_p]),
    "gpdla_objective": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int32, ctypes.c_int32] + [ctypes.c_void_p] * 6),
    "gpdla_objective_device": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int32, ctypes.c_int32] + [ctypes.c_void_p] * 7),
    "gpdla_objective_lyseries": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int32, ctypes.c_int32] + [ctypes.c_void_p] * 3
                                 + [ctypes.c_int32, c_double_p, c_double_p] + [ctypes.c_void_p] * 3),
    "gpdla_objective_lyseries_device": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int32, ctypes.c_int32] + [ctypes.c_void_p] * 3
                                        + [ctypes.c_int32, c_double_p, c_double_p] + [ctypes.c_void_p] * 4),
    "gpdla_default_preload_parameters": (None, [ctypes.POINTER(GpdlaPreloadParams)]),
    "gpdla_preload_qsos": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int64] + [ctypes.c_void_p] * 7
                           + [ctypes.POINTER(GpdlaPreloadParams), ctypes.c_int64] + [ctypes.c_void_p] * 7),
    "gpdla_preload_qsos_device": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int64] + [ctypes.c_void_p] * 7
                                  + [ctypes.POINTER(GpdlaPreloadParams), ctypes.c_int64] + [ctypes.c_void_p] * 8),
    "gpdla_training_set": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int64] + [ctypes.c_void_p] * 7
                           + [ctypes.c_int32, ctypes.c_double, ctypes.c_double] + [ctypes.c_void_p] * 6),
    "gpdla_training_set_device": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int64] + [ctypes.c_void_p] * 7
                                  + [ctypes.c_int32, ctypes.c_double, ctypes.c_double] + [ctypes.c_void_p] * 7),
    "gpdla_pairwise_covariance": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int32] + [ctypes.c_void_p] * 3),
    "gpdla_pairwise_covariance_device": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int32] + [ctypes.c_void_p] * 4),
    "gpdla_training_set_lyseries": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int64] + [ctypes.c_void_p] * 7
                                    + [ctypes.c_int32, ctypes.c_double, ctypes.c_double, ctypes.c_int32]
                                    + [ctypes.c_void_p] * 7),
    "gpdla_training_set_lyseries_device": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int64] + [ctypes.c_void_p] * 7
                                           + [ctypes.c_int32, ctypes.c_double, ctypes.c_double, ctypes.c_int32]
                                           + [ctypes.c_void_p] * 8),
    "gpdla_row_nanmedian_fill": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int32] + [ctypes.c_void_p] * 2),
    "gpdla_row_nanmedian_fill_device": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int32] + [ctypes.c_void_p] * 3),
    "gpdla_dla_statistics": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int64] + [ctypes.c_void_p] * 8
                             + [ctypes.c_int32, c_double_p, ctypes.c_int32, c_double_p, ctypes.c_double, ctypes.c_double,
                                ctypes.c_void_p]),
    "gpdla_dla_statistics_device": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int64] + [ctypes.c_void_p] * 8
                                    + [ctypes.c_int32, c_double_p, ctypes.c_int32, c_double_p, ctypes.c_double,
                                       ctypes.c_double, ctypes.c_void_p, ctypes.c_void_p]),
    "gpdla_multi_dla_statistics": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int64, ctypes.c_int32] + [ctypes.c_void_p] * 9
                                   + [ctypes.c_int32, c_double_p, ctypes.c_int32, c_double_p, ctypes.c_double,
                                      ctypes.c_double, ctypes.c_void_p]),
    "gpdla_multi_dla_statistics_device": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int64, ctypes.c_int32]
                                          + [ctypes.c_void_p] * 9
                                          + [ctypes.c_int32, c_double_p, ctypes.c_int32, c_double_p, ctypes.c_double,
                                             ctypes.c_double, ctypes.c_void_p, ctypes.c_void_p]),
    "gpdla_dla_posteriors": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int64] + [ctypes.c_void_p] * 5
                             + [ctypes.c_int32, c_double_p, ctypes.c_double, ctypes.c_void_p]),
    "gpdla_dla_posteriors_device": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int64] + [ctypes.c_void_p] * 5
                                    + [ctypes.c_int32, c_double_p, ctypes.c_double, ctypes.c_void_p, ctypes.c_void_p]),
    "gpdla_multi_dla_posteriors": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int64, ctypes.c_int32] + [ctypes.c_void_p] * 7),
    "gpdla_multi_dla_posteriors_device": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int64, ctypes.c_int32]
                                          + [ctypes.c_void_p] * 8),
    "gpdla_multi_dla_posterior_quantiles": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int64, ctypes.c_int32]
                                            + [ctypes.c_void_p] * 6
                                            + [ctypes.c_int32, c_double_p, ctypes.c_double, ctypes.c_void_p]),
    "gpdla_multi_dla_posterior_quantiles_device": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int64, ctypes.c_int32]
                                                   + [ctypes.c_void_p] * 6
                                                   + [ctypes.c_int32, c_double_p, ctypes.c_double, ctypes.c_void_p,
                                                      ctypes.c_void_p]),
    "gpdla_reconstruct": (ctypes.c_int,[ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64] + [ctypes.c_void_p] * 6
                          + [ctypes.c_int32, ctypes.c_int32, ctypes.c_void_p, ctypes.c_void_p,
                             ctypes.POINTER(GpdlaReconstruction)]),
    "gpdla_reconstruct_device": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64] + [ctypes.c_void_p] * 6
                                 + [ctypes.c_int32, ctypes.c_int32, ctypes.c_void_p, ctypes.c_void_p,
                                    ctypes.POINTER(GpdlaReconstruction), ctypes.c_void_p]),
    "gpdla_draw_spectra": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64] + [ctypes.c_void_p] * 6
                           + [ctypes.POINTER(GpdlaDrawOptions), ctypes.POINTER(GpdlaDrawOutputs)]),
    "gpdla_draw_spectra_device": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64] + [ctypes.c_void_p] * 6
                                  + [ctypes.POINTER(GpdlaDrawOptions), ctypes.POINTER(GpdlaDrawOutputs),
                                     ctypes.c_void_p]),
}

_lib = None


def load() -> ctypes.CDLL:
    """Load libgpdla.so and bind every declared symbol; raises if the library is not built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                "libgpdla.so is not built (%s). Run `python -c 'import __graft_entry__ as g; g.build()'` or "
                "`python -m gp_dla_detection_b200.build`; gp_dla_detection_b200 has no CPU fallback." % LIB_PATH)
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(lib, name)       # AttributeError if the ABI lost a symbol
            fn.restype, fn.argtypes = res, args
        _lib = lib
    return _lib


class GpdlaError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__("libgpdla error %d: %s" % (code, msg))
        self.code = code


def check(rc: int, ctx=None):
    if rc != GPDLA_OK:
        msg = load().gpdla_last_error(ctx)
        raise GpdlaError(rc, msg.decode() if msg else "")
