#!/usr/bin/env python
"""Benchmark of the per-quasar DLA model-selection hot path (BASELINE.json metric: QSO spectra/s,
10 000 DLA samples each).

  python bench.py --gpus N --steps K --warmup W            our CUDA path (one rank per GPU under torchrun)
  python bench.py --impl reference --steps K --warmup W    the reference algorithm on the host cores
  python bench.py ... --dump-outputs DIR                   also write the last timed step's results as DIR/<name>.npy

A step is one pass of the hot path over this rank's shard of the synthetic catalogue
(BASELINE.json configs[1]: 10 000 DR12Q-shaped quasars per GPU, single-DLA model, k = 20,
10 000 samples, 3 Lyman lines).  The inputs are seeded, so two builds given the same arguments see the same
catalogue and their dumped outputs can be compared array by array.  Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True   # the source tree may be read-only: leave no bytecode caches in it
sys.path.insert(0, ROOT)

METRIC = "qso_spectra_per_sec_10k_dla_samples"
UNIT = "quasars/s"
K_RANK, NUM_SAMPLES, NUM_LINES = 20, 10000, 3


def fp64_peak():
    """FP64 tensor (DMMA) peak in TFLOP/s: MEASURED_PEAKS.json carries no FP64 figure, so the
    denominator is this repo's own step-0 microbenchmark on the same B200 pool."""
    p = os.path.join(ROOT, "profiles", "r01_step0_fp64_peaks.json")
    try:
        return json.load(open(p))["dmma884_cps8_tflops"], "profiles/r01_step0_fp64_peaks.json (mma.sync m8n8k4 f64, measured)"
    except Exception:
        return 37.0, "nominal HGX B200 FP64 tensor (fallback)"


def ncu_traffic(i8):
    """DRAM bytes of one fused log-likelihood launch (296-quasar batch) from the committed ncu --set full capture."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "r02h_ncu_loglik_i8_full.json" if i8 else "r02_ncu_loglik_ws_full.json")))
        return d["dram_bytes_per_launch"], d["Grid Size"]["value"]
    except Exception:
        return None, None


class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.QUERY,
                                       "--format=csv,noheader,nounits", "-lms", "200"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(5)
        except Exception:
            self.p.kill()
        self.f.flush(); self.f.seek(0)
        sm, mx, reasons = [], [], set()
        for line in self.f.read().splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1])); mx.append(float(c[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.f.name)
        if sm:
            out = {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                   "samples": len(sm)}
        return out


def cpu_baseline(model, samples, prior, spectra, n_quasars, threads):
    """The oracle's C restatement of the reference algorithm (process_qsos.m per-sample loop with
    voigt.c + log_mvnpdf_low_rank.m arithmetic), threaded over samples like the reference's parfor."""
    from oracle import process_qsos_oracle as O
    sp = {k: v[:n_quasars] for k, v in spectra.items()}
    t0 = time.perf_counter()
    O.process_qsos(model, samples, sp, prior, num_lines=NUM_LINES, engine="c", nthreads=threads)
    dt = time.perf_counter() - t0
    return n_quasars / dt, dt


def run_reference(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    from gp_dla_detection_b200 import synthetic as syn
    threads = os.cpu_count() or 1
    model = syn.make_model(K_RANK)
    samples = syn.make_samples(NUM_SAMPLES)
    prior = syn.make_prior()
    per_step = args.ref_quasars_per_step
    spectra = syn.make_spectra(model, per_step * (args.steps + args.warmup))
    q0 = 0
    for _ in range(args.warmup):
        cpu_baseline(model, samples, prior, {k: v[q0:q0 + per_step] for k, v in spectra.items()}, per_step, threads)
        q0 += per_step
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_baseline(model, samples, prior, {k: v[q0:q0 + per_step] for k, v in spectra.items()}, per_step, threads)
        q0 += per_step
    dt = time.perf_counter() - t0
    value = per_step * args.steps / dt
    sample = "%d quasars x %d samples per step (bounded sample of the 10000-quasar workload)" % (per_step, NUM_SAMPLES)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "configs[1]: 10000 synthetic DR12Q-shaped quasars, single-DLA, k=20, 10000 samples, "
                               "3 Lyman lines", "sample": sample,
                   "note": "CPU arm: runs on rank 0's host cores only, whatever --gpus says"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
                         "note": "C restatement of process_qsos.m + voigt.c + log_mvnpdf_low_rank.m (oracle/c), "
                                 "OpenMP over samples like the reference's parfor; MATLAB/Octave/libcerf are absent"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def spot_check(proc, model, samples, prior, spectra, timed_out, nq, threads):
    """The CPU restatement on the first `nq` quasars of the timed workload against (a) the outputs of the timed device
    run itself and (b) a fresh call that also returns the sample log-likelihoods.  north_star: same MAP sample,
    log-likelihoods within 1e-8 relative, p_dla within 1e-6 absolute.  Returns (cpu quasars/s, seconds, block)."""
    from oracle import process_qsos_oracle as O
    sp = {k: v[:nq] for k, v in spectra.items()}
    t0 = time.perf_counter()
    ref = O.process_qsos(model, samples, sp, prior, num_lines=NUM_LINES, engine="c", nthreads=threads)
    dt = time.perf_counter() - t0
    got = proc.process(sp, return_sample_log_likelihoods=True)
    rel = lambda a, b: float(np.nanmax(np.abs(np.asarray(a) - np.asarray(b)) / np.abs(np.asarray(b))))
    timed = {k: v[:nq].cpu().numpy() for k, v in timed_out.items()}
    block = {
        "quasars": nq,
        "max_rel_sample_ll": rel(got["sample_log_likelihoods_dla"], ref["sample_log_likelihoods_dla"]),
        "max_rel_ll": max(rel(timed[k], ref[k]) for k in ("log_likelihoods_dla", "log_likelihoods_no_dla",
                                                          "log_posteriors_dla", "log_posteriors_no_dla")),
        "same_map": bool(np.array_equal(timed["map_inds"], ref["map_inds"])),
        "max_abs_p_dla": float(np.nanmax(np.abs(timed["p_dlas"] - ref["p_dlas"]))),
        "timed_run_equals_fresh_call": bool(all(np.array_equal(timed[k], got[k], equal_nan=True) for k in timed)),
        "against": "oracle/c (C restatement of process_qsos.m + voigt.c + log_mvnpdf_low_rank.m), same inputs",
    }
    block["ok"] = bool(block["max_rel_sample_ll"] < 1e-8 and block["max_rel_ll"] < 1e-8 and block["same_map"]
                       and block["max_abs_p_dla"] < 1e-6)
    return nq / dt, dt, block


DUMP_LIMIT_BYTES = 64 * 10 ** 6


def dump_outputs(out, path):
    """Write the arrays a caller of the timed path receives (CUDA tensors, one row per quasar) as path/<name>.npy in
    float64; map_inds (int64 sample indices < 2^53) converts exactly.  When all rows together exceed
    DUMP_LIMIT_BYTES, a fixed seeded sample of rows is written instead, with its row numbers in sampled_quasars.npy."""
    host = {name: t.cpu().numpy().astype(np.float64) for name, t in out.items()}
    Q = len(next(iter(host.values())))
    keep = DUMP_LIMIT_BYTES // (sum(a[:1].nbytes for a in host.values()) + 8)   # + 8: the row number
    os.makedirs(path, exist_ok=True)
    if Q > keep:
        rows = np.sort(np.random.default_rng(0).choice(Q, size=keep, replace=False))
        host = {name: a[rows] for name, a in host.items()}
        host["sampled_quasars"] = rows.astype(np.float64)
    for name, a in host.items():
        np.save(os.path.join(path, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--quasars", type=int, default=10000, help="quasars per GPU per step (configs[1])")
    ap.add_argument("--ref-quasars-per-step", type=int, default=8)
    ap.add_argument("--cpu-baseline-quasars", type=int, default=8)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--gram-digits", type=int, default=0, choices=[-1, 0, 5, 6],
                    help="Gram arithmetic: 0 default (INT8 tensor-core path, 6 digits), -1 FP64 DMMA, 5/6 INT8 digits")
    ap.add_argument("--alt-steps", type=int, default=1,
                    help="timed steps of the secondary leg on the FP64 DMMA Gram (gram_digits = -1); 0 = skip")
    ap.add_argument("--strong-steps", type=int, default=1,
                    help="timed passes of the strong-scaling leg (configs[2]: 162 861 quasars split over the ranks); 0 = skip")
    ap.add_argument("--catalog-quasars", type=int, default=162861, help="size of the full catalogue (configs[2])")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the results of the last one (rank 0's shard) as DIR/<name>.npy, "
                         "float64, at most 64 MB in all")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the results of the CUDA path")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from gp_dla_detection_b200 import api, sharding, synthetic as syn

    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    distributed = world > 1
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # stdout carries the one JSON line and nothing else: native libraries (NCCL prints its version banner there) get
    # stderr as their file descriptor 1 for the whole run; the JSON line goes to the saved descriptor at the end
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    if distributed:
        dist.init_process_group("nccl", device_id=dev)

    # ---- synthetic catalogue shard (weak scaling: args.quasars per GPU), model, samples, prior
    Q = args.quasars
    model = syn.make_model(K_RANK)
    samples = syn.make_samples(NUM_SAMPLES)
    prior = syn.make_prior()
    spectra = syn.make_spectra(model, Q, shard=rank)
    pad = api.pad_spectra(spectra)
    L_max = pad["wavelengths"].shape[1]
    n_used = sharding.quasar_costs(pad)      # pixels in the modelled window per quasar
    masked_in = np.array([np.count_nonzero(np.asarray(m)[(w / (1 + z) >= 911.75) & (w / (1 + z) <= 1215.75)])
                          for w, m, z in zip(spectra["all_wavelengths"], spectra["all_pixel_mask"], spectra["z_qsos"])])
    n_pix = n_used - masked_in               # used pixels n_q
    flops_q = n_pix * float(NUM_SAMPLES * K_RANK * (K_RANK + 3))   # SURVEY 8(d): n k (k+3) per sample
    flops_per_step = float(np.sum(flops_q))

    proc = api.DLAProcessor(model, samples, prior, device=local_rank, gram_digits=args.gram_digits)
    host = {k: torch.from_numpy(np.ascontiguousarray(v)).pin_memory() for k, v in pad.items()}
    dtens = {k: v.to(dev) for k, v in host.items()}
    order = ("wavelengths", "flux", "noise_variance", "pixel_mask", "lengths", "z_qsos")

    def barrier():
        if distributed:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_device(p, tensors, steps):
        """`steps` passes of the device-resident path, CUDA events on the launching stream, max over ranks."""
        barrier()
        p.set_profiling(True)
        p.profile_read()
        n0 = p.launch_count
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            o = p.process_device(*[tensors[k] for k in order])
        e1.record()
        barrier()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if distributed:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        k_ms, k_n = p.profile_read()
        p.set_profiling(False)
        return float(t.item()), o, p.launch_count - n0, k_ms, k_n

    # ---- device-resident timing (inputs already in HBM)
    for _ in range(args.warmup):
        proc.process_device(*[dtens[k] for k in order])
    sampler = ClockSampler(local_rank) if rank == 0 else None
    ms, out, launches, k_ms, k_n = timed_device(proc, dtens, args.steps)
    clocks = sampler.stop() if sampler else None
    value = world * Q * args.steps / (ms * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(out, args.dump_outputs)

    # ---- end to end through the public API: pinned host buffers in, host results out, every step
    hnp = {k: v.numpy() for k, v in host.items()}

    def timed_e2e(want_sll):
        for _ in range(2):
            proc.process(hnp, return_sample_log_likelihoods=want_sll, pinned_results=True)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            r = proc.process(hnp, return_sample_log_likelihoods=want_sll, pinned_results=True)
        torch.cuda.synchronize()
        te = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if distributed:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        return world * Q * args.steps / float(te.item()), r

    e2e_value, res = timed_e2e(False)
    e2e_full_value, res_full = timed_e2e(True)
    h2d = int(sum(hnp[k].nbytes for k in order))
    d2h = int(Q * (14 * 8 + 8))
    d2h_full = d2h + int(Q * NUM_SAMPLES * 8)
    full_equal = bool(all(np.array_equal(res[k], res_full[k], equal_nan=True) for k in res))
    del res_full

    # ---- secondary leg: the FP64 DMMA Gram (the arithmetic north_star names literally), same workload
    alt = None
    if args.alt_steps > 0 and args.gram_digits != -1:
        proc64 = api.DLAProcessor(model, samples, prior, device=local_rank, gram_digits=-1)
        proc64.process_device(*[dtens[k] for k in order])
        ms64, out64, _, k64_ms, k64_n = timed_device(proc64, dtens, args.alt_steps)
        peak, _ = fp64_peak()
        ach = flops_per_step * args.alt_steps / (k64_ms * 1e-3) * 1e-12
        a, b = out64["log_likelihoods_dla"].cpu().numpy(), out["log_likelihoods_dla"].cpu().numpy()
        alt = {"gram_arithmetic": "FP64 DMMA (mma.sync m8n8k4 f64), dla_loglik_ws_kernel", "steps": args.alt_steps,
               "value": world * Q * args.alt_steps / (ms64 * 1e-3), "unit": UNIT, "ms_per_step": ms64 / args.alt_steps,
               "roofline": {"bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
                            "kernel_ms_per_step": k64_ms / args.alt_steps, "kernel_launches": int(k64_n)},
               "max_rel_log_likelihoods_dla_vs_primary": float(np.nanmax(np.abs(a - b) / np.abs(b)))}
        proc64.close()
        del proc64, out64

    # ---- strong-scaling leg: configs[2], the full catalogue split across the ranks (no data-path collective)
    strong = None
    if args.strong_steps > 0:
        Qcat = args.catalog_quasars
        # the catalogue is the 10 000-quasar synthetic shard of rank 0's seed repeated; contiguous blocks balanced by
        # cost (pixels in the modelled window), as sharding.partition_by_cost does for a real catalogue
        base = api.pad_spectra(syn.make_spectra(model, Q, shard=0)) if rank != 0 else pad
        idx = np.arange(Qcat) % Q
        blocks = sharding.partition_by_cost(sharding.quasar_costs(base)[idx], world)
        b0, b1 = blocks[rank]
        sel = torch.from_numpy(idx[b0:b1]).to(dev)
        bt = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in base.items()} if rank != 0 else dtens
        cat = {k: bt[k].index_select(0, sel).contiguous() for k in order}
        ms_s, out_s, _, _, _ = timed_device(proc, cat, args.strong_steps)
        strong = {"workload": "configs[2]: %d-quasar synthetic catalogue (the %d-quasar shard repeated), quasars split "
                              "across %d rank(s) by cost" % (Qcat, Q, world),
                  "value": Qcat * args.strong_steps / (ms_s * 1e-3), "unit": UNIT, "scaling": "strong",
                  "seconds_per_catalogue": ms_s * 1e-3 / args.strong_steps, "steps": args.strong_steps,
                  "quasars_this_rank": int(b1 - b0)}
        del cat, out_s

    # ---- multi-GPU: the one collective of the path, a gather of per-quasar records (outside the hot loop)
    if distributed:
        rec = sharding.pack_records({k: v for k, v in res.items()})
        blocks = [(r * Q, (r + 1) * Q) for r in range(world)]
        full = sharding.gather_records(rec, blocks, device=dev)
        assert full.shape == (world * Q, sharding.RECORD_WIDTH)

    ok = True
    if rank == 0:
        peak, peak_src = fp64_peak()
        achieved = flops_per_step * args.steps / (k_ms * 1e-3) * 1e-12 if k_ms > 0 else None
        digits = args.gram_digits if args.gram_digits != 0 else 6
        i8 = digits in (5, 6)
        traffic, traffic_grid = ncu_traffic(i8)
        roof = {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                "frac": (achieved / peak) if achieved else None, "traffic": traffic,
                "traffic_note": "dram__bytes_read+write of one launch with grid %s (one 296-quasar batch; this "
                                "run launches the same batch size), ncu --set full, profiles/r02_ncu_loglik_*_full.json" % traffic_grid,
                "algorithmic_flops_per_launch": flops_per_step * args.steps / max(int(k_n), 1),
                "kernel_ms_per_step": k_ms / args.steps, "kernel_launches": int(k_n),
                "kernel_share_of_step": k_ms / ms,
                "timed_interval": "CUDA events on the launching stream around each batch's fused kernels: the persistent INT8 "
                                  "kernel on 132 SMs and, concurrently on the 16 SMs its clusters cannot occupy, the FP64 DMMA "
                                  "kernel on the last 7 % of the batch (second stream, joined before the interval ends)",
                "algorithmic_flops_per_step": flops_per_step, "peak_source": peak_src,
                "peak_nominal": 40.0, "peak_nominal_source": "NVIDIA HGX B200 datasheet, FP64 tensor, per GPU"}
        if i8:
            # int8 operations the tcgen05 MMAs execute: per cluster (128 samples) and 32-pixel chunk, L(L+1)/2 slice
            # pairs x (3 CTAs x N=80 + 1 CTA x N=32) columns x 128 rows x 32 pixels x 2
            pairs = digits * (digits + 1) // 2
            chunks = np.sum((n_used + 31) // 32)
            clusters = (NUM_SAMPLES + 1 + 127) // 128
            int8_ops = float(chunks) * clusters * pairs * 2.0 * 128 * 32 * (3 * 80 + 32)
            roof.update({
                "kernel": "dla_loglik_i8p_kernel (fused optical depth from a rest-frame table + instrument convolution + "
                          "exact-product INT8 tcgen05 Gram, %d signed 8-bit digits per factor, s32 TMEM accumulators + "
                          "Cholesky; persistent 4-CTA clusters, two-stage producer warp pairs, DSMEM row-block exchange, "
                          "epilogue warpgroup, merged slice-pair MMAs, MN-major digit tiles)" % digits,
                "note": "achieved/peak = FP64-equivalent Gram rate (S n k(k+3) per quasar, SURVEY 8(d)) over the "
                        "builder-measured FP64 DMMA peak (MEASURED_PEAKS.json has no FP64 entry; nominal 40 beside it); "
                        "the contraction itself runs as exact INT8 slice products on the tcgen05 tensor pipe, see "
                        "int8_tensor. On B200 FP64 arithmetic makes no progress while a tcgen05.mma executes on the "
                        "same SM (profiles/r01_mma_vs_alu.json; ncu: sm__pipe_shared = fp64 + tensor), so a 32-pixel "
                        "chunk costs the producers' FP64 work plus the tensor time of the 21 exact slice products "
                        "(DESIGN.md 4.3-4.4). 132 of the 148 SMs host clusters (4-CTA cluster placement)",
                "int8_tensor": {"achieved_tops": int8_ops * args.steps / (k_ms * 1e-3) * 1e-12 if k_ms > 0 else None,
                                "peak_tops": 4283.0, "peak_source": "profiles/r01_tcgen05_i8.txt (this pool's B200, N = 240)"},
            })
        else:
            roof.update({
                "kernel": "dla_loglik_ws_kernel (fused Voigt + FP64 DMMA Gram + Cholesky, warp-specialised)",
                "note": "FP64 DMMA and DFMA share one pipe on B200 (measured): the fused kernel's Voigt/"
                        "weight arithmetic competes with the Gram for the same 37 TFLOP/s"})
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "configs[1]: %d synthetic DR12Q-shaped quasars per GPU, single-DLA, k=%d, %d "
                                   "samples, %d Lyman lines, L_max=%d" % (Q, K_RANK, NUM_SAMPLES, NUM_LINES, L_max),
                       "quasars_per_gpu": Q, "l2": "inputs %.0f MB + per-batch workspace > 126 MB L2; no flush needed"
                                                   % (h2d / 1e6),
                       "gram_arithmetic": ("exact-product int8 x int8 -> s32 slices of FP64 operands, %d digits (%d "
                                           "fractional bits)" % (digits, 8 * digits - 1)) if i8 else "FP64 DMMA",
                       "sharding": "quasars split across ranks, no data-path collective; one all_gather of records"},
            "gpu_launches": int(launches),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "note": "DLAProcessor.process: pinned host planes in, the 15 per-quasar result columns out"},
            "e2e_full": {"value": e2e_full_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h_full,
                         "note": "the same call returning sample_log_likelihoods_dla as well (process_qsos.m:236-244 saves "
                                 "it): 80 KB per quasar into a page-locked buffer, batch t copied while batch t + 1 computes",
                         "other_outputs_equal_e2e": full_equal},
            "roofline": roof,
            "clocks": clocks,
        }
        if alt is not None:
            line["alt"] = alt
        if strong is not None:
            line["strong"] = strong
        if not args.no_cpu_baseline:
            threads = os.cpu_count() or 1
            nq = args.cpu_baseline_quasars
            v, dt, block = spot_check(proc, model, samples, prior, spectra, out, nq, threads)
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
                                    "sample": "%d quasars x %d samples of the same workload (%.1f s)" % (nq, NUM_SAMPLES, dt)}
            line["parity_spot"] = block
            ok = block["ok"]
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    if distributed:
        dist.destroy_process_group()
    if not ok:
        sys.stderr.write("bench.py: the timed outputs disagree with the CPU restatement beyond north_star's tolerance\n")
        sys.exit(1)


if __name__ == "__main__":
    main()
