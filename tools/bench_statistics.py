"""Population-statistics sums (gpdla_dla_statistics_device) on one GPU vs the host route:
python tools/bench_statistics.py [num_quasars] [out.json]   -> one JSON object (recorded under profiles/).

Workload: synthetic.make_spectra(make_model(), Q, dla_fraction=0.3) through DLAProcessor.process_device with the
10 000 default samples, then the statistics of that batch with 5 z bins and 30 log-N bins.  At Q = 20 000 the sample
log-likelihoods are 1.6 GB, larger than the 126 MB L2, so every timed pass reads them from HBM.  Device-event times,
after warm-up, averaged over repeated launches, of (a) the statistics entry and (b) process_device of the same batch.
The host route is what the entry replaces: the device-to-host copy of the likelihoods (timed) plus the NumPy
restatement on one core, timed on a subset of quasars and scaled to Q (it is linear in Q)."""
import json, os, subprocess, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from gp_dla_detection_b200 import api, synthetic as syn
from oracle import dla_statistics_oracle as O

Q = int(sys.argv[1]) if len(sys.argv) > 1 else 20000
OUT = sys.argv[2] if len(sys.argv) > 2 else None
S, reps, warm, host_subset = 10000, 10, 3, 40
HBM_TBS = 7.7                # TB/s, HBM3e bandwidth of one B200 (data sheet)
Z_EDGES = np.linspace(2.0, 5.0, 6)
N_EDGES = np.linspace(20.0, 23.0, 31)


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


t0 = time.perf_counter()
model = syn.make_model()
samples = syn.make_samples(S)
spectra = syn.make_spectra(model, Q, dla_fraction=0.3)
pad = api.pad_spectra(spectra)
gen_s = time.perf_counter() - t0
dev = torch.device("cuda", 0)
up = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dtype=dt)).to(dev)
planes = (up(pad["wavelengths"], np.float64), up(pad["flux"], np.float64), up(pad["noise_variance"], np.float64),
          up(pad["pixel_mask"], np.uint8), up(pad["lengths"], np.int32), up(pad["z_qsos"], np.float64))
proc = api.DLAProcessor(model, samples, syn.make_prior(), device=0)
out = proc.process_device(*planes, return_sample_log_likelihoods=True)
process_ms = timed(lambda: proc.process_device(*planes, return_sample_log_likelihoods=True, out=out), n=2, w=1)
sums = torch.zeros(api.dla_statistics_width(5, 30), dtype=torch.float64, device=dev)


def run_stats():
    sums.zero_()
    proc.statistics_device(out, Z_EDGES, N_EDGES, sums=sums)


zero_ms = timed(lambda: sums.zero_())
stats_ms = timed(run_stats)
first = sums.cpu().numpy().copy()                  # the sums of one call
run_stats(); torch.cuda.synchronize()
repeat = bool(first.tobytes() == sums.cpu().numpy().tobytes())
# where the time goes: one call under torch.profiler, a run of its own after the timed window
from torch.profiler import profile, ProfilerActivity
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    run_stats()
    torch.cuda.synchronize()
kernel_us = {k.key: k.device_time_total for k in prof.key_averages() if k.device_time_total > 0}
# host route: D2H of the likelihoods and per-quasar results, then the restatement
t0 = time.perf_counter()
host = {k: v.cpu().numpy() for k, v in out.items()}
d2h_s = time.perf_counter() - t0
t0 = time.perf_counter()
sub = O.dla_statistics_sums(host["sample_log_likelihoods_dla"][:host_subset], host["p_dlas"][:host_subset],
                            host["min_z_dlas"][:host_subset], host["max_z_dlas"][:host_subset],
                            samples["offset_samples"], samples["log_nhi_samples"], samples["nhi_samples"], Z_EDGES,
                            N_EDGES)
oracle_subset_s = time.perf_counter() - t0
got_sub = api.dla_statistics_sums({k: v[:host_subset] for k, v in host.items()}, samples, Z_EDGES, N_EDGES)
g, r = api.unpack_dla_statistics(got_sub, 5, 30), api.unpack_dla_statistics(sub, 5, 30)
nz = lambda x: np.maximum(np.abs(x), 1e-300)
sub_err = max(float(np.max(np.abs(g[k] - r[k]) / nz(r[k]))) for k in ("counts", "dla", "nhi", "path"))
# q (1 - q) cancels where q is near 1: its error is measured against the mean it comes from
var_err = max(float(np.max(np.abs(g[k] - r[k]) / nz(r[k] + r[m]))) for k, m in (("counts_var", "counts"),
                                                                                  ("dla_var", "dla")))
W = api.dla_statistics_width(5, 30)
contributing = int(round(first[-1]))
stat_bytes = Q * S * 8 + Q * (3 * 8) + 2 * Q * W * 8 + S * 8 * 3
finished = api.finish_dla_statistics(first, Z_EDGES, N_EDGES)
res = {
    "workload": "%d synthetic quasars (dla_fraction 0.3) x %d samples, 5 z bins on [2, 5], 30 log-N bins on [20, 23]; "
                "%d quasars contribute; sample_log_likelihoods_dla %.2f GB (larger than L2)"
                % (Q, S, contributing, Q * S * 8 / 1e9),
    "gpu": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit_max_sm_clock": power_limit(),
    "timing": "CUDA events, %d warm-up + %d timed launches, back to back on one stream; statistics_ms has the "
              "zeroing of the 2 KB sums vector (zero_ms) subtracted" % (warm, reps),
    "statistics_ms": stats_ms - zero_ms, "zero_ms": zero_ms,
    "statistics_note": "per call: sample class + rank sort (S^2 comparisons) + gather, one CTA per quasar (staged row, "
                       "one exp per sample, binary searches, fixed-order cell sums), fixed-block column sums, finish",
    "statistics_bytes": stat_bytes, "statistics_hbm_bound_ms": stat_bytes / (HBM_TBS * 1e12) * 1e3,
    "statistics_bytes_note": "likelihood rows + per-quasar scalars read once, per-quasar cell rows written and read "
                             "once, samples",
    "statistics_exp_count": Q * S,
    "kernel_us_one_profiled_call": kernel_us,
    "process_device_ms_same_batch": process_ms,
    "statistics_fraction_of_process": (stats_ms - zero_ms) / process_ms,
    "host_route_d2h_s": d2h_s,
    "host_route_oracle_s_on_%d_quasars" % host_subset: oracle_subset_s,
    "host_route_oracle_s_scaled_to_Q": oracle_subset_s * Q / host_subset,
    "host_route_note": "one core; the NumPy restatement loops per sample and is timed on a subset, scaled linearly",
    "repeat_bit_identical": repeat,
    "max_rel_err_vs_oracle_%d_quasars_counts_dla_nhi_path" % host_subset: sub_err,
    "max_err_vs_oracle_%d_quasars_variances_over_var_plus_mean" % host_subset: var_err,
    "dndx": finished["dndx"].tolist(), "omega_dla": finished["omega_dla"].tolist(),
    "host_generation_s": gen_s,
}
proc.close()
text = json.dumps(res, indent=1)
print(text)
if OUT:
    with open(OUT, "w") as fh:
        fh.write(text + "\n")
