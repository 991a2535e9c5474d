"""Credible intervals of every absorber of the multi-DLA model (gpdla_multi_dla_posterior_quantiles_device) on one GPU:
python tools/bench_multi_posterior_quantiles.py [out.json]   -> one JSON object (recorded under profiles/).

Workload, that of the multi-DLA section of tools/bench_posteriors.py: synthetic.make_spectra(make_model(), 2000,
dla_fraction=0.3, meanflux=True, second_dla_fraction=0.3) through process_multi_device once (that call is timed) with
J = 4 and 10 000 samples, tiled 10x to 20 000 quasars, 5 quantiles (api.DEFAULT_QUANTILES).  The rows and partner
indices are 8.8 GB, far larger than the 126 MB L2, so every timed call reads them from HBM.  Device-event times of 3
warm-up and 10 timed calls, for this entry and for multi_posteriors_device on the same input; the outputs are checked
against the NumPy restatement on a subset of quasars, every deviation named by its field."""
import json, os, subprocess, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from gp_dla_detection_b200 import api, synthetic as syn
from oracle import dla_posteriors_oracle as O
from oracle import multi_dla_posterior_quantiles_oracle as MQ

OUT = sys.argv[1] if len(sys.argv) > 1 else None
Q0, TILE, S, J, reps, warm, subset = 2000, 10, 10000, 4, 10, 3, 24
HBM_TBS = 7.7                # TB/s, HBM3e bandwidth of one B200 (data sheet)
QS = api.DEFAULT_QUANTILES
P = len(QS)


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=60)
        return r.stdout.strip() or r.stderr.strip()
    except Exception as e:              # the number is still valid; say why the limit is missing
        return "unavailable: %s" % e


def timed(fn):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


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


def deviations(got, ll, part, zlo, zhi, off, lnhi):
    """Per field (mass_above_threshold, z_quantiles, log_nhi_quantiles): the largest |got - restatement| and where it
    is, and for the quantiles how many lie outside the values the restatement's cumulative sums allow at
    MQ.quantile_tolerance(S)."""
    ref = MQ.multi_dla_posterior_quantiles(ll, part, zlo, zhi, off, lnhi, QS)
    g, r = (api.unpack_multi_dla_posterior_quantiles(x, J, P) for x in (got, ref))
    out = {"nan_patterns_equal": bool(np.array_equal(np.isnan(got), np.isnan(ref)))}
    for name in ("mass_above_threshold", "z_quantiles", "log_nhi_quantiles"):
        d = np.abs(g[name] - r[name])
        d[~np.isfinite(d)] = 0.0
        at = np.unravel_index(int(np.argmax(d)), d.shape)
        out[name] = {"max_abs_dev": float(d[at]),
                     "at_quasar_level_rank" + ("_p" if d.ndim == 4 else ""): [int(at[0]), int(at[1]) + 1]
                     + [int(x) for x in at[2:]]}
    tol, outside, ambiguous = MQ.quantile_tolerance(S), 0, 0
    for q in range(ll.shape[0]):
        for j in range(1, J + 1):
            w = O.weights(ll[q, j - 1])
            if w is None or not np.isfinite(g["z_quantiles"][q, j - 1, 0, 0]):
                continue
            z, n = O.ranked_slots(part[q], j, zlo[q], zhi[q], off, lnhi)
            for rk in range(j):
                for name, vals in (("z_quantiles", z[rk]), ("log_nhi_quantiles", n[rk])):
                    for k, p in enumerate(QS):
                        ok, amb = O.acceptable_quantiles(vals, w, p, tol)
                        outside += g[name][q, j - 1, rk, k] not in ok
                        ambiguous += amb
    out["quantiles_outside_acceptable_set"] = outside
    out["quantiles_with_more_than_one_acceptable_value"] = ambiguous
    out["tolerance"] = tol
    return out


dev = torch.device("cuda", 0)
up = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dtype=dt)).to(dev)
t0 = time.perf_counter()
res = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit_max_sm_clock": card(),
       "timing": "CUDA events, %d warm-up + %d timed calls back to back on one stream" % (warm, reps)}
model = syn.make_model()
samples = syn.make_samples(S, with_lls=True)
pad = api.pad_spectra(syn.make_spectra(model, Q0, dla_fraction=0.3, meanflux=True, second_dla_fraction=0.3))
planes = (up(pad["wavelengths"], np.float64), up(pad["flux"], np.float64), up(pad["noise_variance"], np.float64),
          up(pad["pixel_mask"], np.uint8), up(pad["lengths"], np.int32), up(pad["z_qsos"], np.float64))
proc = api.DLAProcessor(model, samples, syn.make_prior(), device=0)
proc.process_multi_device(*(t[:200] for t in planes), max_dlas=J, return_samples=True)   # workspaces, tables
out, process_ms = once(lambda: proc.process_multi_device(*planes, max_dlas=J, return_samples=True))
names = ("sample_log_likelihoods_dla", "base_sample_inds", "min_z_dlas", "max_z_dlas")
tiled = {k: out[k].repeat((TILE,) + (1,) * (out[k].dim() - 1)).contiguous() for k in names}
del out
Q = Q0 * TILE
moments_ms = timed(lambda: proc.multi_posteriors_device(tiled))
quant_ms = timed(lambda: proc.multi_posterior_quantiles_device(tiled, QS))
moments_ms_after = timed(lambda: proc.multi_posteriors_device(tiled))   # the spread of the reference
first = proc.multi_posterior_quantiles_device(tiled, QS).cpu().numpy()
repeat = bool(first.tobytes() == proc.multi_posterior_quantiles_device(tiled, QS).cpu().numpy().tobytes())
kernel_us = profiled(lambda: proc.multi_posterior_quantiles_device(tiled, QS))
host = {k: tiled[k][:subset].cpu().numpy() for k in names}
dev_check = deviations(first[:subset], host["sample_log_likelihoods_dla"], host["base_sample_inds"],
                       host["min_z_dlas"], host["max_z_dlas"], samples["offset_samples"], samples["log_nhi_samples"])
proc.close()
nbytes = Q * J * S * 8 + Q * (J - 1) * S * 4 + Q * 2 * 8 + Q * api.multi_dla_posterior_quantiles_width(J, P) * 8
hbm_ms = nbytes / (HBM_TBS * 1e12) * 1e3
t = api.unpack_multi_dla_posterior_quantiles(first, J, P)
res["multi_quantiles"] = {
    "workload": "%d synthetic mean-flux quasars (dla_fraction 0.3, second_dla_fraction 0.3) through process_multi_device "
                "(J = %d, %d samples), tiled %dx to %d quasars, %d quantiles; rows + partner indices %.2f GB (larger "
                "than L2)" % (Q0, J, S, TILE, Q, P, (Q * J * S * 8 + Q * (J - 1) * S * 4) / 1e9),
    "posterior_quantiles_ms": quant_ms,
    "multi_posteriors_ms_before_and_after": [moments_ms, moments_ms_after],
    "times_multi_posteriors": quant_ms / (0.5 * (moments_ms + moments_ms_after)),
    "process_multi_device_ms_%d_quasars_one_call" % Q0: process_ms,
    "process_multi_device_ms_scaled_to_%d" % Q: process_ms * TILE,
    "fraction_of_process_multi_device": quant_ms / (process_ms * TILE),
    "bytes": nbytes, "hbm_bound_ms": hbm_ms, "times_hbm_bound": quant_ms / hbm_ms,
    "bytes_note": "likelihood rows (J S doubles) and partner indices ((J - 1) S int32) read once per quasar, min/max z "
                  "read and records written once; the 10 sample passes per quasar re-read the rows from L2 or HBM",
    "kernel_us_one_profiled_call": kernel_us,
    "repeat_bit_identical": repeat,
    "vs_oracle_first_%d_quasars" % subset: dev_check,
    "finite_levels_1_to_%d" % J: np.count_nonzero(np.isfinite(t["mass_above_threshold"][:, :, 0]), axis=0).tolist(),
}
res["card_after"] = card()
res["host_s"] = time.perf_counter() - t0
text = json.dumps(res, indent=1)
print(text)
if OUT:
    with open(OUT, "w") as fh:
        fh.write(text + "\n")
