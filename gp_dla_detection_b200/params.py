"""Parameters of the DLA detection pipeline -- mirror of the reference's ``set_parameters.m``.

Same names as the MATLAB workspace variables (set_parameters.m:5-73) so that code and tests
read like the reference; only the entries the per-quasar hot path uses are kept.
"""
from __future__ import annotations

from dataclasses import dataclass

lya_wavelength = 1215.6701          # set_parameters.m:5   Lyman alpha transition wavelength (A)
lyb_wavelength = 1025.7223          # :6
lyman_limit = 911.7633              # :7
speed_of_light = 299792458.0        # :8   m/s


def kms_to_z(kms: float) -> float:  # set_parameters.m:11
    return (kms * 1000.0) / speed_of_light


@dataclass(frozen=True)
class Parameters:
    """Hot-path parameters (defaults = the reference's DR12Q configuration)."""
    min_lambda: float = 911.75                        # :33  null-model rest-wavelength range (A)
    max_lambda: float = 1215.75                       # :34
    dlambda: float = 0.25                             # :35
    k: int = 20                                       # :36  rank of the low-rank covariance term
    num_dla_samples: int = 10000                      # :48
    prior_z_qso_increase: float = kms_to_z(30000.0)   # :56
    width: int = 3                                    # :59  instrument-profile half width (pixels)
    pixel_spacing: float = 1e-4                       # :60  dex
    num_lines: int = 3                                # :63  Lyman-series members in the DLA profile
    max_z_cut: float = kms_to_z(3000.0)               # :65
    min_z_cut: float = kms_to_z(3000.0)               # :69
    min_num_pixels: int = 200                         # :26
    z_qso_cut: float = 2.15                           # :25
    loading_min_lambda: float = 910.0                 # :15
    loading_max_lambda: float = 1217.0                # :16
    max_noise_variance: float = 1.0 ** 2              # next to k: noisier interpolated pixels leave the training set
    initial_c_0: float = 0.1                          # :40  starting point of the null-model fit
    initial_tau_0: float = 0.0023                     # :41
    initial_beta: float = 3.65                        # :42


DEFAULT = Parameters()
