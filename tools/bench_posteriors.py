"""Per-quasar absorber posterior summaries (gpdla_dla_posteriors_device, gpdla_multi_dla_posteriors_device) on one GPU:
python tools/bench_posteriors.py [out.json]   -> one JSON object (recorded under profiles/).

Workloads, each through its processing entry once (that call is timed) and tiled 10x to 20 000 quasars:
- single-DLA: synthetic.make_spectra(make_model(), 2000, dla_fraction=0.3) through process_device, 10 000 default
  samples, 5 quantiles (api.DEFAULT_QUANTILES);
- multi-DLA: make_spectra(..., meanflux=True, second_dla_fraction=0.3) through process_multi_device with J = 4.
At 20 000 quasars the rows are 1.6 GB (single) and 6.4 GB + 2.4 GB of partner indices (multi), far larger than the
126 MB L2, so every timed call reads them from HBM.  Device-event times of 3 warm-up and 10 timed calls; the timed
outputs are checked against the NumPy restatement on a subset of quasars."""
import json, os, subprocess, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from gp_dla_detection_b200 import api, synthetic as syn
from oracle import dla_posteriors_oracle as O

OUT = sys.argv[1] if len(sys.argv) > 1 else None
Q0, TILE, S, J, reps, warm, subset = 2000, 10, 10000, 4, 10, 3, 24
HBM_TBS = 7.7                # TB/s, HBM3e bandwidth of one B200 (data sheet)
QS = api.DEFAULT_QUANTILES


def card():
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
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n


def once(fn):
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    r = fn()
    b.record()
    torch.cuda.synchronize()
    return r, a.elapsed_time(b)


def profiled(fn):
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {k.key: k.device_time_total for k in prof.key_averages() if k.device_time_total > 0}


def err_over_scale(got, ref, mean_of):
    """max |got - ref| / (|ref| + floor) over the entries finite in both, NaN when the NaN patterns differ.  A standard
    deviation or covariance (column c, mean_of[c] its means' columns) is known to the rounding of the values, so its
    floor is 4e-16 times the scale of its means, as in tests/test_dla_posteriors.py."""
    if not np.array_equal(np.isfinite(ref), np.isfinite(got)):
        return float("nan")
    floor = np.zeros_like(ref)
    for c, means in mean_of.items():
        floor[:, c] = 4e-16 * np.prod(np.abs(ref[:, means]), axis=1) ** (1.0 / len(means))
    f = np.isfinite(ref)
    return float(np.max(np.abs(got[f] - ref[f]) / np.maximum(np.abs(ref[f]) + floor[f], 1e-300))) if f.any() else 0.0


dev = torch.device("cuda", 0)
up = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dtype=dt)).to(dev)
model = syn.make_model()
card_before = card()
res = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit_max_sm_clock": card_before,
       "timing": "CUDA events, %d warm-up + %d timed calls back to back on one stream" % (warm, reps)}

# ---- single-DLA
t0 = time.perf_counter()
samples = syn.make_samples(S, with_lls=True)
pad = api.pad_spectra(syn.make_spectra(model, Q0, dla_fraction=0.3))
planes = (up(pad["wavelengths"], np.float64), up(pad["flux"], np.float64), up(pad["noise_variance"], np.float64),
          up(pad["pixel_mask"], np.uint8), up(pad["lengths"], np.int32), up(pad["z_qsos"], np.float64))
proc = api.DLAProcessor(model, samples, syn.make_prior(), device=0)
proc.process_device(*(t[:200] for t in planes), return_sample_log_likelihoods=True)   # workspaces, tables
out, process_ms = once(lambda: proc.process_device(*planes, return_sample_log_likelihoods=True))
names = ("sample_log_likelihoods_dla", "min_z_dlas", "max_z_dlas")
tiled = {k: out[k].repeat((TILE,) + (1,) * (out[k].dim() - 1)).contiguous() for k in names}
del out
Q = Q0 * TILE
post_ms = timed(lambda: proc.posteriors_device(tiled, QS))
first = proc.posteriors_device(tiled, QS).cpu().numpy()
repeat = bool(first.tobytes() == proc.posteriors_device(tiled, QS).cpu().numpy().tobytes())
kernel_us = profiled(lambda: proc.posteriors_device(tiled, QS))
host = {k: tiled[k][:subset].cpu().numpy() for k in names}
ref = O.dla_posteriors(host["sample_log_likelihoods_dla"], host["min_z_dlas"], host["max_z_dlas"],
                       samples["offset_samples"], samples["log_nhi_samples"], QS)
single_bytes = Q * S * 8 + Q * 2 * 8 + Q * api.dla_posteriors_width(len(QS)) * 8
res["single"] = {
    "workload": "%d synthetic quasars (dla_fraction 0.3) through process_device (%d samples), tiled %dx to %d "
                "quasars, %d quantiles; rows %.2f GB (larger than L2)" % (Q0, S, TILE, Q, len(QS), Q * S * 8 / 1e9),
    "posteriors_ms": post_ms,
    "process_device_ms_%d_quasars_one_call" % Q0: process_ms,
    "process_device_ms_scaled_to_%d" % Q: process_ms * TILE,
    "posteriors_fraction_of_process": post_ms / (process_ms * TILE),
    "bytes": single_bytes, "hbm_bound_ms": single_bytes / (HBM_TBS * 1e12) * 1e3,
    "times_hbm_bound": post_ms / (single_bytes / (HBM_TBS * 1e12) * 1e3),
    "bytes_note": "likelihood rows read once, min/max z read and records written once",
    "kernel_us_one_profiled_call": kernel_us,
    "repeat_bit_identical": repeat,
    "max_err_vs_oracle_%d_quasars_over_scale" % subset: err_over_scale(first[:subset], ref, {2: [1], 4: [3], 5: [1, 3]}),
    "finite_records": int(np.count_nonzero(np.isfinite(first[:, 0]))),
    "ess_percentiles_5_50_95": np.nanpercentile(first[:Q0, 0], [5, 50, 95]).tolist(),
}
proc.close()
del tiled
torch.cuda.empty_cache()

# ---- multi-DLA
pad = api.pad_spectra(syn.make_spectra(model, Q0, dla_fraction=0.3, meanflux=True, second_dla_fraction=0.3))
planes = (up(pad["wavelengths"], np.float64), up(pad["flux"], np.float64), up(pad["noise_variance"], np.float64),
          up(pad["pixel_mask"], np.uint8), up(pad["lengths"], np.int32), up(pad["z_qsos"], np.float64))
proc = api.DLAProcessor(model, samples, syn.make_prior(), device=0)
proc.process_multi_device(*(t[:200] for t in planes), max_dlas=J, return_samples=True)
out, mprocess_ms = once(lambda: proc.process_multi_device(*planes, max_dlas=J, return_samples=True))
names = ("sample_log_likelihoods_dla", "base_sample_inds", "min_z_dlas", "max_z_dlas")
tiled = {k: out[k].repeat((TILE,) + (1,) * (out[k].dim() - 1)).contiguous() for k in names}
del out
mpost_ms = timed(lambda: proc.multi_posteriors_device(tiled))
mfirst = proc.multi_posteriors_device(tiled).cpu().numpy()
mrepeat = bool(mfirst.tobytes() == proc.multi_posteriors_device(tiled).cpu().numpy().tobytes())
mkernel_us = profiled(lambda: proc.multi_posteriors_device(tiled))
host = {k: tiled[k][:subset].cpu().numpy() for k in names}
mref = O.multi_dla_posteriors(host["sample_log_likelihoods_dla"], host["base_sample_inds"], host["min_z_dlas"],
                              host["max_z_dlas"], samples["offset_samples"], samples["log_nhi_samples"])
multi_bytes = Q * J * S * 8 + Q * (J - 1) * S * 4 + Q * 2 * 8 + Q * api.multi_dla_posteriors_width(J) * 8
proc.close()
res["multi"] = {
    "workload": "%d synthetic mean-flux quasars (dla_fraction 0.3, second_dla_fraction 0.3) through process_multi_device "
                "(J = %d, %d samples), tiled %dx to %d quasars; rows + partner indices %.2f GB (larger than L2)"
                % (Q0, J, S, TILE, Q, (Q * J * S * 8 + Q * (J - 1) * S * 4) / 1e9),
    "posteriors_ms": mpost_ms,
    "process_multi_device_ms_%d_quasars_one_call" % Q0: mprocess_ms,
    "process_multi_device_ms_scaled_to_%d" % Q: mprocess_ms * TILE,
    "posteriors_fraction_of_process": mpost_ms / (mprocess_ms * TILE),
    "bytes": multi_bytes, "hbm_bound_ms": multi_bytes / (HBM_TBS * 1e12) * 1e3,
    "times_hbm_bound": mpost_ms / (multi_bytes / (HBM_TBS * 1e12) * 1e3),
    "bytes_note": "likelihood rows and partner indices read once, min/max z read and records written once",
    "kernel_us_one_profiled_call": mkernel_us,
    "repeat_bit_identical": mrepeat,
    "max_err_vs_oracle_%d_quasars_over_scale" % subset: err_over_scale(
        mfirst[:subset], mref, {c: [c - 1] for j in range(1, J + 1) for r in range(j)
                                for c in (j - 1 + 2 * (j - 1) * j + 2 + 4 * r, j - 1 + 2 * (j - 1) * j + 4 + 4 * r)}),
    "finite_records_per_level": np.count_nonzero(np.isfinite(api.unpack_multi_dla_posteriors(mfirst, J)["ess"]),
                                                 axis=0).tolist(),
}
res["card_after"] = card()
res["host_s"] = time.perf_counter() - t0
text = json.dumps(res, indent=1)
print(text)
if OUT:
    with open(OUT, "w") as fh:
        fh.write(text + "\n")
