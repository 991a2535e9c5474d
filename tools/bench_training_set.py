"""Training set + PCA initialisation (learn_qso_model.m:36-95) on one GPU vs the NumPy restatement on the host:
python tools/bench_training_set.py [num_spectra] [out.json]   -> one JSON object (recorded under profiles/).

Workload: synthetic.make_spectra(make_model(), N, dla_fraction=0), P = 1217 rest pixels, k = 20.  Device-event times,
after warm-up, averaged over repeated launches, of (a) gpdla_training_set_device (interpolation kernel + column
reductions) and (b) gpdla_pairwise_covariance_device (column means + DMMA tile kernel + fixed-order finish).  At
N = 20 000 the centred matrix is 195 MB, larger than the 126 MB L2, so every timed pass reads it from HBM."""
import ctypes, json, os, subprocess, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from gp_dla_detection_b200 import _lib, api, synthetic as syn
from gp_dla_detection_b200.params import DEFAULT, lya_wavelength
from oracle import training_set_oracle as TS

N = int(sys.argv[1]) if len(sys.argv) > 1 else 20000
OUT = sys.argv[2] if len(sys.argv) > 2 else None
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
sp = syn.make_spectra(syn.make_model(), N, dla_fraction=0)
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
