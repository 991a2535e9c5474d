"""Draws from the learned model (gpdla_draw_spectra_device) on one GPU:
python tools/bench_draw_spectra.py [num_quasars] [out.json]   -> one JSON object (recorded under profiles/).

Workload: the observing setups of synthetic.make_spectra(make_model(20), Q) with 10 000 samples, in four
configurations: prior-predictive draws of the single-DLA model, of the multi-DLA model (max_dlas = 4), a draw with 4
given absorbers per quasar under the mean-flux null model, and the injection of 4 given absorbers into the batch's
flux.  The absorption plane is not requested (the flux is the product).  Device-event times averaged over 10 calls
after 3 of warm-up, plus one process_device call on the same batch for scale, and the host time per quasar of
make_spectra at Q = 500 (the CPU generator the tests used so far).

Bounds from shapes: bytes = the planes read (wavelength and noise variance as float64, mask as uint8, and the flux when
injecting) and the flux written, per pixel of the padded batch; the prior catalogue (read by every CTA of a prior draw)
stays in L2 and is not counted.  FP64 operations = 2 per multiply-add of M~ xi (k per window pixel, draws only) and,
per absorber and padded window pixel, ~30 per line for the optical depth plus 16 for the exponential and the 7-tap
sum; the null model's interpolation, the forest model, Box-Muller and the integer Philox rounds are not counted, so the
operation bound is a lower bound."""
import json, os, subprocess, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from gp_dla_detection_b200 import api, synthetic as syn
from gp_dla_detection_b200 import params as P

Q = int(sys.argv[1]) if len(sys.argv) > 1 else 20000
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
t0 = time.perf_counter()
syn.make_spectra(model, 500, seed=1, dla_fraction=0.3)
make_spectra_us = (time.perf_counter() - t0) / 500 * 1e6
spectra = syn.make_spectra(model, Q, dla_fraction=0.3)
pad = api.pad_spectra(spectra)
L_max = pad["wavelengths"].shape[1]
dev = torch.device("cuda", 0)
up = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dtype=dt)).to(dev)
planes = (up(pad["wavelengths"], np.float64), up(pad["flux"], np.float64), up(pad["noise_variance"], np.float64),
          up(pad["pixel_mask"], np.uint8), up(pad["lengths"], np.int32), up(pad["z_qsos"], np.float64))
n_win = np.zeros(Q)
z4 = np.empty((Q, 4))
for q in range(Q):
    lam, z = spectra["all_wavelengths"][q], spectra["z_qsos"][q]
    win = (lam / (1 + z) >= P.DEFAULT.min_lambda) & (lam / (1 + z) <= P.DEFAULT.max_lambda)
    n_win[q] = np.count_nonzero(win)
    lo, hi = lam[win].min() / P.lya_wavelength - 1, lam[win].max() / P.lya_wavelength - 1
    z4[q] = lo + (hi - lo) * np.array([0.15, 0.4, 0.65, 0.9])
az, an = up(z4, np.float64), up(np.full((Q, 4), 10.0 ** 20.8), np.float64)

proc = api.DLAProcessor(model, samples, syn.make_prior(), device=0)
torch.cuda.synchronize()
process_ms = timed(lambda: proc.process_device(*planes), n=1, w=1)

workloads = [("single prior", dict(model="single"), False),
             ("multi prior (max_dlas 4)", dict(model="multi", max_dlas=4), False),
             ("draw, 4 given absorbers, mean-flux model", dict(model="multi", absorber_z=az, absorber_nhi=an), False),
             ("inject 4 given absorbers", dict(model="single", inject=True, absorber_z=az, absorber_nhi=an), True)]
results = []
for name, kw, inject in workloads:
    draw = proc.draw_spectra_device(*planes, seed=1, return_absorption=False, **kw)
    torch.cuda.synchronize()
    if "truth_model" in draw:       # absorbers actually placed, for the operation count
        codes = draw["truth_model"].cpu().numpy()
        A = np.where(codes >= 2, codes - 1, np.where(codes == 1, 1, 0))
    else:
        A = np.full(Q, 4)
    ms = timed(lambda: proc.draw_spectra_device(*planes, seed=1, return_absorption=False, **kw))
    bytes_ = Q * L_max * (2 * 8 + 1 + 8 + (8 if inject else 0)) + Q * (4 + 8) + (Q * 4 * 16 if "absorber_z" in kw else 0)
    flops = (0 if inject else 2 * K * n_win.sum()) + (A * (n_win + 6)).sum() * (30 * P.DEFAULT.num_lines + 16)
    t_hbm, t_fp64 = bytes_ / (HBM_TBS * 1e12) * 1e3, flops / (FP64_TFLOPS * 1e12) * 1e3
    results.append(dict(workload=name, ms=ms, us_per_quasar=ms * 1e3 / Q, mean_absorbers=float(A.mean()),
                        hbm_bytes=bytes_, fp64_ops=float(flops), hbm_bound_ms=t_hbm, fp64_bound_ms=t_fp64,
                        nearer_bound="fp64" if t_fp64 > t_hbm else "hbm", ratio_to_nearer_bound=ms / max(t_hbm, t_fp64),
                        share_of_process_device=ms / process_ms))
proc.close()
line = dict(tool="bench_draw_spectra", device=torch.cuda.get_device_name(0), nvidia_smi=power_limit(), Q=Q, k=K,
            num_samples=10000, L_max=L_max, mean_window_pixels=float(n_win.mean()), reps=reps, warmup=warm,
            process_device_ms=process_ms, make_spectra_host_us_per_quasar=make_spectra_us, hbm_tbs=HBM_TBS,
            fp64_tflops=FP64_TFLOPS, results=results)
s = json.dumps(line, indent=1)
print(s)
if OUT:
    os.makedirs(os.path.dirname(os.path.abspath(OUT)), exist_ok=True)
    with open(OUT, "w") as f:
        f.write(s + "\n")
