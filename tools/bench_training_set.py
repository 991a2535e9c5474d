"""Training set + PCA initialisation (learn_qso_model.m:36-95) on one GPU vs the NumPy restatement on the host:
python tools/bench_training_set.py [--meanflux] [num_spectra] [out.json]   -> one JSON object (recorded under profiles/).

Workload: synthetic.make_spectra(make_model(), N, dla_fraction=0), P = 1217 rest pixels, k = 20.  Device-event times,
after warm-up, averaged over repeated launches, of (a) gpdla_training_set_device (interpolation kernel + column
reductions) and (b) gpdla_pairwise_covariance_device (column means + DMMA tile kernel + fixed-order finish).  At
N = 20 000 the centred matrix is 195 MB, larger than the 126 MB L2, so every timed pass reads it from HBM.

--meanflux: the multi-DLA model's training set (learn_qso_model_meanflux.m) on meanflux=True spectra instead, timing
separately (a) gpdla_training_set_lyseries_device with 31 Lyman-series members (kernel + column reductions), (b)
gpdla_row_nanmedian_fill_device and (c) gpdla_pairwise_covariance_device on the filled matrix, each against its bound."""
import ctypes, json, os, subprocess, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from gp_dla_detection_b200 import _lib, api, params, synthetic as syn
from gp_dla_detection_b200.params import DEFAULT, MULTI, lya_wavelength
from oracle import training_set_meanflux_oracle as MF
from oracle import training_set_oracle as TS

MEANFLUX = "--meanflux" in sys.argv
argv = [a for a in sys.argv[1:] if a != "--meanflux"]
N = int(argv[0]) if len(argv) > 0 else 20000
OUT = argv[1] if len(argv) > 1 else None
k, reps, warm = 20, 10, 3
DMMA_PEAK = 36.997          # TFLOP/s, m8n8k4 at 8 CTAs/SM on a B200 (profiles/r01_step0_fp64_peaks.json)


def power_limit():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=60)
        return r.stdout.strip() or r.stderr.strip()
    except Exception as e:              # the number is still valid; say why the limit is missing
        return "unavailable: %s" % e


t0 = time.perf_counter()
sp = syn.make_spectra(syn.make_model(), N, dla_fraction=0, meanflux=MEANFLUX)
pad = api.pad_spectra(sp)
gen_s = time.perf_counter() - t0
dev = torch.device("cuda", 0)
up = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
W, F, V = up(pad["wavelengths"]), up(pad["flux"]), up(pad["noise_variance"])
Mk, lengths, z = up(pad["pixel_mask"].astype(np.uint8)), up(pad["lengths"].astype(np.int32)), up(pad["z_qsos"])
L_max = W.shape[1]
rest = api.rest_wavelengths()
P = rest.size
f64 = dict(dtype=torch.float64, device=dev)
rest_d = up(rest)
lya, y, nv = (torch.empty((N, P), **f64) for _ in range(3))
mu, sd = torch.empty(P, **f64), torch.empty(P, **f64)
nobs = torch.empty(P, dtype=torch.int32, device=dev)
cov = torch.empty((P, P), **f64)
counts = torch.empty((P, P), dtype=torch.int32, device=dev)
lib = _lib.load()
ptr = lambda t: ctypes.c_void_p(t.data_ptr())
stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def run_training_set():
    _lib.check(lib.gpdla_training_set_device(N, L_max, ptr(W), ptr(F), ptr(V), ptr(Mk), ptr(lengths), ptr(z), ptr(rest_d),
                                             P, lya_wavelength, DEFAULT.max_noise_variance, ptr(lya), ptr(y), ptr(nv),
                                             ptr(mu), ptr(sd), ptr(nobs), stream))


def run_covariance():
    _lib.check(lib.gpdla_pairwise_covariance_device(N, P, ptr(y), ptr(cov), ptr(counts), stream))


def timed(fn):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


HBM_TBS = 7.7                # TB/s, HBM3e bandwidth of one B200 (data sheet)


def run_meanflux():
    """--meanflux: three stages timed separately, each against its bound; returns the JSON object."""
    nl = params.num_forest_lines
    absorption, filled = torch.empty((N, P), **f64), torch.empty((N, P), **f64)

    def run_lyseries():
        _lib.check(lib.gpdla_training_set_lyseries_device(
            N, L_max, ptr(W), ptr(F), ptr(V), ptr(Mk), ptr(lengths), ptr(z), ptr(rest_d), P, lya_wavelength,
            MULTI.max_noise_variance, nl, ptr(lya), ptr(y), ptr(nv), ptr(absorption), ptr(mu), ptr(sd), ptr(nobs), stream))

    def run_fill():
        _lib.check(lib.gpdla_row_nanmedian_fill_device(N, P, ptr(y), ptr(filled), stream))

    def run_cov_filled():
        _lib.check(lib.gpdla_pairwise_covariance_device(N, P, ptr(filled), ptr(cov), ptr(counts), stream))

    plain_ms = timed(run_training_set)       # the single-DLA build on the same spectra, for comparison
    ts_ms = timed(run_lyseries)              # leaves y = the centred fluxes of one build
    fill_ms = timed(run_fill)
    cov_ms = timed(run_cov_filled)
    # repeatability of the three stages
    y1, f1, c1 = y.clone(), filled.clone(), cov.clone()
    run_lyseries(); run_fill(); run_cov_filled(); torch.cuda.synchronize()
    repeat = bool(torch.equal(y.nan_to_num(7.0), y1.nan_to_num(7.0)) and torch.equal(filled.nan_to_num(7.0), f1.nan_to_num(7.0))
                  and torch.equal(cov, c1))
    # executed pow calls: the Lya term of every kept pixel plus each member l >= 1 where 1 + z_l <= 1 + z_qso, counted
    # from lya_1pzs scaled by lambda_Lya / lambda_l (equal to the kernel's 1 + z_l up to rounding)
    kept = ~torch.isnan(lya)
    opz = (1.0 + z)[:, None]
    tw = params.all_transition_wavelengths
    pows = int(kept.sum())
    for l in range(1, nl):
        pows += int((kept & (lya * (lya_wavelength / tw[l]) <= opz)).sum())
    observed = int(kept.sum())
    NP = N * P
    ts_bytes = N * L_max * (3 * 8 + 1) + N * 12 + 4 * NP * 8 + 4 * NP * 8   # planes in, 4 matrices out, 3 reductions
    fill_bytes = 2 * NP * 8
    nrows = int(((~torch.isnan(y)).sum(dim=1).gt(0) & torch.isnan(y).any(dim=1)).sum())
    S = 1 << (P - 1).bit_length()
    stages = S.bit_length() - 1
    stages = stages * (stages + 1) // 2
    sort_smem_bytes = nrows * stages * S * 8 * 2       # every stage loads S keys and stores up to S
    smi = power_limit()
    try:
        sm_mhz = float(smi.split(",")[2].strip().split()[0])
    except Exception:
        sm_mhz = float("nan")
    smem_tbs = 148 * 128 * sm_mhz * 1e6 * 1e-12       # 128 B per clock per SM at the maximum SM clock
    tiles = (P + 63) // 64
    flops = P * (P + 1) / 2 * N * 2.0
    # oracle spot check of the fill on a fixed sample of rows of the GPU's centred matrix
    rows = np.random.default_rng(0).choice(N, 256, replace=False)
    yh = y[rows].cpu().numpy()
    fill_equal = bool(np.array_equal(filled[rows].cpu().numpy(), MF.row_nanmedian_fill(yh), equal_nan=True))
    return {
        "workload": "learn_qso_model_meanflux.m: %d synthetic meanflux spectra (dla_fraction 0, L_max %d) x %d rest "
                    "pixels, %d Lyman-series members, max_noise_variance %g, %.1f %% of the centred matrix observed"
                    % (N, L_max, P, nl, MULTI.max_noise_variance, 100.0 * float((~torch.isnan(y)).sum()) / NP),
        "gpu": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit_max_sm_clock": smi,
        "timing": "CUDA events, %d warm-up + %d timed launches each, back to back on one stream" % (warm, reps),
        "training_set_lyseries_ms": ts_ms, "training_set_plain_ms_same_spectra": plain_ms,
        "training_set_lyseries_note": "interpolation + 31-member mean-flux correction kernel + 3 column reductions",
        "training_set_bytes": ts_bytes, "training_set_hbm_bound_ms": ts_bytes / (HBM_TBS * 1e12) * 1e3,
        "training_set_executed_pow": pows, "training_set_pow_per_kept_pixel": pows / observed,
        "training_set_pow_note": "Lya term of every kept pixel + members l >= 1 with 1 + z_l <= 1 + z_qso, counted on "
                                 "the host from lya_1pzs (equal to the kernel's count up to rounding at the boundary); "
                                 "31 per kept pixel without the skip",
        "median_fill_ms": fill_ms, "median_fill_bytes": fill_bytes,
        "median_fill_hbm_bound_ms": fill_bytes / (HBM_TBS * 1e12) * 1e3,
        "median_fill_rows_sorted": nrows, "median_fill_sort_size": S, "median_fill_network_stages": stages,
        "median_fill_sort_shared_bytes": sort_smem_bytes,
        "median_fill_shared_bound_ms": sort_smem_bytes / (smem_tbs * 1e12) * 1e3,
        "median_fill_shared_bound_note": "shared-memory traffic of the bitonic network at 128 B per clock per SM, 148 "
                                         "SMs, the maximum SM clock above",
        "covariance_filled_ms": cov_ms, "covariance_flop": flops, "covariance_tflops": flops / (cov_ms * 1e-3) * 1e-12,
        "covariance_executed_flop": tiles * (tiles + 1) / 2 * 64 * 64 * N * 2.0,
        "covariance_dmma_bound_ms": tiles * (tiles + 1) / 2 * 64 * 64 * N * 2.0 / (DMMA_PEAK * 1e12) * 1e3,
        "dmma_peak_tflops_measured": DMMA_PEAK, "hbm_tb_per_s_datasheet": HBM_TBS,
        "repeat_bit_identical": repeat, "median_fill_equals_oracle_on_256_rows": fill_equal,
        "host_generation_s": gen_s,
    }


if MEANFLUX:
    text = json.dumps(run_meanflux(), indent=1)
    print(text)
    if OUT:
        with open(OUT, "w") as fh:
            fh.write(text + "\n")
    sys.exit(0)

ts_ms = timed(run_training_set)           # leaves y = the centred fluxes of one build (the build overwrites, not adds)
cov_ms = timed(run_covariance)
cov_h, std_h = cov.cpu().numpy(), sd.cpu().numpy()
cov_again = cov.clone(); run_covariance(); torch.cuda.synchronize()
t0 = time.perf_counter(); w, _ = np.linalg.eigh(cov_h); eigh_s = time.perf_counter() - t0
x0 = api._initial_x(cov_h, std_h, k, rest, DEFAULT)
# the host restatement of the same build (steps 1-6)
t0 = time.perf_counter(); ref = TS.training_set(sp, k); oracle_s = time.perf_counter() - t0
ok = ~np.isnan(ref["cov"])
flops = P * (P + 1) / 2 * N * 2.0
tflops = flops / (cov_ms * 1e-3) * 1e-12
tiles = (P + 63) // 64
res = {
    "workload": "learn_qso_model.m:36-95: %d synthetic spectra (dla_fraction 0, L_max %d) x %d rest pixels, k = %d, "
                "%.1f %% of the centred matrix observed" % (N, L_max, P, k, 100.0 * float((~torch.isnan(y)).sum()) / (N * P)),
    "gpu": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit_max_sm_clock": power_limit(),
    "training_set_ms": ts_ms, "training_set_spectra_per_s": N / ts_ms * 1e3,
    "training_set_note": "interpolation kernel + 3 column reductions (mean, centring, nanstd) over the [N x P] matrices",
    "covariance_ms": cov_ms, "covariance_flop": flops, "covariance_tflops": tflops,
    "covariance_fraction_of_dmma_peak": tflops / DMMA_PEAK, "dmma_peak_tflops_measured": DMMA_PEAK,
    "covariance_executed_flop": tiles * (tiles + 1) / 2 * 64 * 64 * N * 2.0,
    "covariance_note": "P(P+1)/2 N 2 FLOP (the lower triangle); the kernel executes %d full 64 x 64 tiles" % (tiles * (tiles + 1) // 2),
    "covariance_repeat_bit_identical": bool(torch.equal(cov_again, cov)),
    "host_eigh_s": eigh_s, "host_oracle_training_set_s": oracle_s, "host_generation_s": gen_s,
    "timing": "CUDA events, %d warm-up + %d timed launches each, back to back on one stream" % (warm, reps),
    "cov_max_abs_err_over_max_vs_oracle": float(np.max(np.abs(cov_h[ok] - ref["cov"][ok])) / np.abs(ref["cov"][ok]).max()),
    "counts_equal_oracle": bool(np.array_equal(counts.cpu().numpy(), ref["counts"])),
    "mu_max_rel_err_vs_oracle": float(np.max(np.abs(mu.cpu().numpy() - ref["mu"]) / np.abs(ref["mu"]))),
    "initial_x_max_abs_err_over_max_vs_oracle": float(np.max(np.abs(x0 - ref["initial_x"])) / np.abs(ref["initial_x"]).max()),
}
text = json.dumps(res, indent=1)
print(text)
if OUT:
    with open(OUT, "w") as fh:
        fh.write(text + "\n")
