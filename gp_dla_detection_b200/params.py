"""Parameters of the DLA detection pipeline -- mirror of the reference's ``set_parameters.m``.

Same names as the MATLAB workspace variables (set_parameters.m:5-73) so that code and tests
read like the reference; only the entries the per-quasar hot path uses are kept.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

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

# ---- the multi-DLA / mean-flux model (multi_dlas/set_parameters_multi.m, learn_qso_model_meanflux.m)
MULTI = Parameters(max_noise_variance=3.0 ** 2)      # set_parameters_multi.m:37; everything else as DEFAULT
prev_tau_0 = 0.0023                                  # learn_qso_model_meanflux.m: Kim et al. (2007) mean-flux prior
prev_beta = 3.65
num_forest_lines = 31                                # set_parameters_multi.m:76
# set_parameters_multi.m:77-109, Angstrom (the cm values of voigt.c times 1e8, as the library computes them)
all_transition_wavelengths = np.array([
    1.2156701e-05, 1.0257223e-05, 9.725368e-06, 9.497431e-06, 9.378035e-06, 9.307483e-06, 9.262257e-06,
    9.231504e-06, 9.209631e-06, 9.193514e-06, 9.181294e-06, 9.171806e-06, 9.16429e-06, 9.15824e-06, 9.15329e-06,
    9.14919e-06, 9.14576e-06, 9.14286e-06, 9.14039e-06, 9.13826e-06, 9.13641e-06, 9.13480e-06, 9.13339e-06,
    9.13215e-06, 9.13104e-06, 9.13006e-06, 9.12918e-06, 9.12839e-06, 9.12768e-06, 9.12703e-06, 9.12645e-06]) * 1e8
all_oscillator_strengths = np.array([                # :111-143
    0.416400, 0.079120, 0.029000, 0.013940, 0.007799, 0.004814, 0.003183, 0.002216, 0.001605, 0.00120, 0.000921,
    0.0007226, 0.000577, 0.000469, 0.000386, 0.000321, 0.000270, 0.000230, 0.000197, 0.000170, 0.000148, 0.000129,
    0.000114, 0.000101, 0.000089, 0.000080, 0.000071, 0.000064, 0.000058, 0.000053, 0.000048])
all_transition_wavelengths.flags.writeable = False
all_oscillator_strengths.flags.writeable = False

# ---- population statistics of the single-DLA catalogue (CDDF_analysis/calc_cddf.py; api.dla_statistics_sums,
# api.finish_dla_statistics).  Flat LambdaCDM with Omega_Lambda = 1 - omega_m and no radiation.  The defaults
# omega_m = 0.3, hubble_h = 0.7 are this package's choice: they are not checked against calc_cddf.py.
omega_m = 0.3
hubble_h = 0.7                                       # H0 = 100 h km/s/Mpc
dla_log_nhi_min = 20.3                               # a sample is a DLA where log10 N_HI >= this
gravitational_constant = 6.67430e-8                  # cm^3 g^-1 s^-2, CODATA 2018
speed_of_light_cgs = 2.99792458e10                   # cm/s
hydrogen_mass = 1.6735575e-24                        # g, m_H (the hydrogen atom; no helium correction anywhere)
megaparsec = 3.0856775814913673e24                   # cm
