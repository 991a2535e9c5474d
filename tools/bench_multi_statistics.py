"""Population-statistics sums of the multi-DLA model (gpdla_multi_dla_statistics_device) on one GPU:
python tools/bench_multi_statistics.py [out.json]   -> one JSON object (recorded under profiles/).

Workload: synthetic.make_spectra(make_model(), 2000, dla_fraction=0.3, meanflux=True, second_dla_fraction=0.3) through
DLAProcessor.process_multi_device once (J = 4, the 10 000 default samples; that call is timed), its outputs tiled to
20 000 quasars, then the statistics of those with 5 z bins and 30 log-N bins.  At 20 000 quasars the rows and partner
indices are 8.8 GB, far larger than the 126 MB L2, so every timed call reads them from HBM.  Device-event times of 3
warm-up and 10 timed calls; the timed output is checked against the NumPy restatement on a subset of quasars."""
import json, os, subprocess, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from gp_dla_detection_b200 import api, synthetic as syn
from oracle import multi_dla_statistics_oracle as O

OUT = sys.argv[1] if len(sys.argv) > 1 else None
Q0, TILE, S, J, reps, warm, subset = 2000, 10, 10000, 4, 10, 3, 24
HBM_TBS = 7.7                # TB/s, HBM3e bandwidth of one B200 (data sheet)
Z_EDGES = np.linspace(2.0, 5.0, 6)
N_EDGES = np.linspace(20.0, 23.0, 31)


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=60)
        return r.stdout.strip() or r.stderr.strip()
    except Exception as e:              # the number is still valid; say why the limit is missing
        return "unavailable: %s" % e


t0 = time.perf_counter()
model = syn.make_model()
samples = syn.make_samples(S, with_lls=True)
spectra = syn.make_spectra(model, Q0, dla_fraction=0.3, meanflux=True, second_dla_fraction=0.3)
pad = api.pad_spectra(spectra)
gen_s = time.perf_counter() - t0
dev = torch.device("cuda", 0)
up = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dtype=dt)).to(dev)
planes = (up(pad["wavelengths"], np.float64), up(pad["flux"], np.float64), up(pad["noise_variance"], np.float64),
          up(pad["pixel_mask"], np.uint8), up(pad["lengths"], np.int32), up(pad["z_qsos"], np.float64))
proc = api.DLAProcessor(model, samples, syn.make_prior(), device=0)
proc.process_multi_device(*(t[:200] for t in planes), max_dlas=J, return_samples=True)   # workspaces, tables
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
out = proc.process_multi_device(*planes, max_dlas=J, return_samples=True)
e1.record()
torch.cuda.synchronize()
process_ms = e0.elapsed_time(e1)
names = ("sample_log_likelihoods_dla", "base_sample_inds", "model_posteriors", "min_z_dlas", "max_z_dlas")
tiled = {k: out[k].repeat((TILE,) + (1,) * (out[k].dim() - 1)).contiguous() for k in names}
Q = Q0 * TILE
del out
sums = torch.zeros(api.dla_statistics_width(5, 30), dtype=torch.float64, device=dev)


def run_stats():
    sums.zero_()
    proc.multi_statistics_device(tiled, Z_EDGES, N_EDGES, sums=sums)


def timed(fn, n=reps, w=warm):
    for _ in range(w):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n


card_before = card()
zero_ms = timed(lambda: sums.zero_())
stats_ms = timed(run_stats) - zero_ms
first = sums.cpu().numpy().copy()
run_stats(); torch.cuda.synchronize()
repeat = bool(first.tobytes() == sums.cpu().numpy().tobytes())
from torch.profiler import profile, ProfilerActivity
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    run_stats()
    torch.cuda.synchronize()
kernel_us = {k.key: k.device_time_total for k in prof.key_averages() if k.device_time_total > 0}
# the timed output against the restatement: the first `subset` quasars (the tiles repeat them)
host = {k: tiled[k][:subset].cpu().numpy() for k in names}
got = proc.multi_statistics_device({k: tiled[k][:subset] for k in names}, Z_EDGES, N_EDGES).cpu().numpy()
t0 = time.perf_counter()
ref = O.multi_dla_statistics_sums(host["sample_log_likelihoods_dla"], host["base_sample_inds"], host["model_posteriors"],
                                  host["min_z_dlas"], host["max_z_dlas"], samples["offset_samples"],
                                  samples["log_nhi_samples"], samples["nhi_samples"], Z_EDGES, N_EDGES)
oracle_s = time.perf_counter() - t0
g, r = api.unpack_dla_statistics(got, 5, 30), api.unpack_dla_statistics(ref, 5, 30)
nz = lambda x: np.maximum(np.abs(x), 1e-300)
mean_err = max(float(np.max(np.abs(g[k] - r[k]) / nz(r[k]))) for k in ("counts", "dla", "nhi", "path"))
var_err = max(float(np.max(np.abs(g[k] - r[k]) / nz(np.abs(r[k]) + 4 * r[m] + r[m] ** 2)))
              for k, m in (("counts_var", "counts"), ("dla_var", "dla")))
W = api.dla_statistics_width(5, 30)
stat_bytes = Q * J * S * 8 + Q * (J - 1) * S * 4 + Q * (J + 4) * 8 + 2 * Q * W * 8 + S * (8 + 8 + 4)
finished = api.finish_dla_statistics(first, Z_EDGES, N_EDGES)
process_same_ms = process_ms * Q / Q0
res = {
    "workload": "%d synthetic mean-flux quasars (dla_fraction 0.3, second_dla_fraction 0.3) through process_multi_device "
                "(J = %d, %d samples), tiled %dx to %d quasars; 5 z bins on [2, 5], 30 log-N bins on [20, 23]; %d "
                "quasars contribute; rows + partner indices %.2f GB (larger than L2)"
                % (Q0, J, S, TILE, Q, int(round(first[-1])), (Q * J * S * 8 + Q * (J - 1) * S * 4) / 1e9),
    "gpu": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit_max_sm_clock": card_before,
    "timing": "CUDA events, %d warm-up + %d timed calls back to back on one stream; the zeroing of the sums vector "
              "(zero_ms) is subtracted" % (warm, reps),
    "multi_statistics_ms": stats_ms, "zero_ms": zero_ms,
    "process_multi_device_ms_%d_quasars_one_call" % Q0: process_ms,
    "process_multi_device_ms_scaled_to_%d" % Q: process_same_ms,
    "multi_statistics_fraction_of_process_multi": stats_ms / process_same_ms,
    "statistics_bytes": stat_bytes, "statistics_hbm_bound_ms": stat_bytes / (HBM_TBS * 1e12) * 1e3,
    "statistics_bytes_note": "likelihood rows and partner indices + per-quasar scalars read once, per-quasar cell rows "
                             "written and read once, samples",
    "times_hbm_bound": stats_ms / (stat_bytes / (HBM_TBS * 1e12) * 1e3),
    "kernel_us_one_profiled_call": kernel_us,
    "repeat_bit_identical": repeat,
    "max_rel_err_vs_oracle_%d_quasars_counts_dla_nhi_path" % subset: mean_err,
    "max_err_vs_oracle_%d_quasars_variances_over_their_scale" % subset: var_err,
    "oracle_s_%d_quasars" % subset: oracle_s,
    "dndx": finished["dndx"].tolist(), "omega_dla": finished["omega_dla"].tolist(),
    "host_generation_s": gen_s,
}
proc.close()
text = json.dumps(res, indent=1)
print(text)
if OUT:
    with open(OUT, "w") as fh:
        fh.write(text + "\n")
