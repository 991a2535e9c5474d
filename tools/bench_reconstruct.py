"""The fitted-model reconstruction (gpdla_reconstruct_device) on one GPU:
python tools/bench_reconstruct.py [num_quasars] [out.json]   -> one JSON object (recorded under profiles/).

Workload: synthetic.make_spectra(make_model(20), Q) with every output requested, in four configurations: 0 and 4
absorbers per quasar (spread over each window), single-DLA and mean-flux null model.  Device-event times averaged over
10 calls after 3 of warm-up, plus one process_device call on the same batch (10 000 samples) for scale.  The inputs
and outputs (about 1 GB at Q = 10 000) exceed the 126 MB L2, so every call reads and writes HBM.

Bounds from shapes: bytes = the planes read (3 float64 + 1 uint8 per pixel) and written (6 float64 per pixel), per
quasar scalars and absorbers; FP64 operations = 2 per multiply-add of the Gram (k+1)(k+2)/2 entries per used pixel, of
the planes (k(k+1)/2 + 3k per window pixel) and, per absorber and padded pixel, ~30 per line for the optical depth
(the wing polynomial and reciprocal) plus 16 for the exponential and the 7-tap sum; interpolation and the forest model
are not counted, so the operation bound is a lower bound."""
import json, os, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from gp_dla_detection_b200 import api, synthetic as syn
from gp_dla_detection_b200 import params as P

Q = int(sys.argv[1]) if len(sys.argv) > 1 else 10000
OUT = sys.argv[2] if len(sys.argv) > 2 else None
K, reps, warm = 20, 10, 3
HBM_TBS = 7.7                # TB/s, HBM3e bandwidth of one B200 (data sheet)
FP64_TFLOPS = 34.0           # DFMA peak measured on the pool's B200 (profiles/r01_step0_fp64_peaks.json)


def power_limit():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=60)
        return r.stdout.strip() or r.stderr.strip()
    except Exception as e:              # the number is still valid; say why the limit is missing
        return "unavailable: %s" % e


def timed(fn, n=reps, w=warm):
    for _ in range(w):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


model = syn.make_model(K)
samples = syn.make_samples(10000, with_lls=True)
spectra = syn.make_spectra(model, Q, dla_fraction=0.3)
pad = api.pad_spectra(spectra)
L_max = pad["wavelengths"].shape[1]
dev = torch.device("cuda", 0)
up = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dtype=dt)).to(dev)
planes = (up(pad["wavelengths"], np.float64), up(pad["flux"], np.float64), up(pad["noise_variance"], np.float64),
          up(pad["pixel_mask"], np.uint8), up(pad["lengths"], np.int32), up(pad["z_qsos"], np.float64))
# window and used pixel counts per quasar (for the bounds)
n_win, n_used = np.zeros(Q), np.zeros(Q)
z4 = np.empty((Q, 4))
for q in range(Q):
    lam, z = spectra["all_wavelengths"][q], spectra["z_qsos"][q]
    win = (lam / (1 + z) >= P.DEFAULT.min_lambda) & (lam / (1 + z) <= P.DEFAULT.max_lambda)
    n_win[q], n_used[q] = np.count_nonzero(win), np.count_nonzero(win & ~spectra["all_pixel_mask"][q])
    lo, hi = lam[win].min() / P.lya_wavelength - 1, lam[win].max() / P.lya_wavelength - 1
    z4[q] = lo + (hi - lo) * np.array([0.15, 0.4, 0.65, 0.9])
n4 = np.full((Q, 4), 10.0 ** 20.8)

proc = api.DLAProcessor(model, samples, syn.make_prior(), device=0)
torch.cuda.synchronize()
process_ms = timed(lambda: proc.process_device(*planes), n=1, w=1)

naug = (K + 1) * (K + 2) / 2
results = []
for meanflux in (False, True):
    for A in (0, 4):
        az = torch.from_numpy(z4[:, :A].copy()).to(dev) if A else None
        an = torch.from_numpy(n4[:, :A].copy()).to(dev) if A else None
        ms = timed(lambda: proc.reconstruct_device(*planes, absorber_z=az, absorber_nhi=an, meanflux=meanflux))
        bytes_ = Q * L_max * (3 * 8 + 1) + Q * L_max * 6 * 8 + Q * (4 + 8 + K * 8 + 8 + 8 + 4) + Q * A * 16
        flops = (2 * naug * n_used.sum() + 2 * (K * (K + 1) / 2 + 3 * K) * n_win.sum()
                 + A * (n_win + 6).sum() * (30 * P.DEFAULT.num_lines + 16))
        t_hbm, t_fp64 = bytes_ / (HBM_TBS * 1e12) * 1e3, flops / (FP64_TFLOPS * 1e12) * 1e3
        results.append(dict(meanflux=meanflux, num_absorbers=A, ms=ms, hbm_bytes=bytes_, fp64_ops=flops,
                            hbm_bound_ms=t_hbm, fp64_bound_ms=t_fp64, nearer_bound="fp64" if t_fp64 > t_hbm else "hbm",
                            ratio_to_nearer_bound=ms / max(t_hbm, t_fp64), share_of_process_device=ms / process_ms))
proc.close()
line = dict(tool="bench_reconstruct", device=torch.cuda.get_device_name(0), nvidia_smi=power_limit(), Q=Q, k=K,
            L_max=L_max, mean_window_pixels=float(n_win.mean()), mean_used_pixels=float(n_used.mean()),
            reps=reps, warmup=warm, process_device_ms=process_ms, hbm_tbs=HBM_TBS, fp64_tflops=FP64_TFLOPS,
            results=results)
s = json.dumps(line, indent=1)
print(s)
if OUT:
    os.makedirs(os.path.dirname(os.path.abspath(OUT)), exist_ok=True)
    with open(OUT, "w") as f:
        f.write(s + "\n")
