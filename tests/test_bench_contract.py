"""bench.py's reference arm runs without a GPU (it times the oracle's C restatement on the host cores): one JSON line
on stdout with the keys a caller reads, the same metric / unit / config as the CUDA arm.  --dump-outputs writes what
the timed CUDA path returned in its last step."""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def load_bench():
    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_reference_arm_prints_one_json_line():
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0", "--ref-quasars-per-step", "1"], capture_output=True, text=True, timeout=600,
                         env=dict(os.environ, RANK="0", WORLD_SIZE="1"))
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "qso_spectra_per_sec_10k_dla_samples" and d["unit"] == "quasars/s"
    assert d["higher_is_better"] is True and d["steps"] == 1 and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "quasars/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_reference_arm_is_silent_on_other_ranks():
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, timeout=120, env=dict(os.environ, RANK="1", WORLD_SIZE="2"))
    assert res.returncode == 0 and res.stdout.strip() == ""


def test_steps_must_be_positive():
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"],
                         capture_output=True, text=True, timeout=120, env=dict(os.environ, RANK="0", WORLD_SIZE="1"))
    assert res.returncode == 2 and "--steps" in res.stderr and res.stdout == ""


def test_dump_outputs_writes_float64_within_the_size_limit(tmp_path, monkeypatch):
    import torch
    bench = load_bench()
    Q = 50
    rng = np.random.default_rng(3)
    out = {"p_dlas": torch.from_numpy(rng.random(Q)), "model_posteriors": torch.from_numpy(rng.random((Q, 2))),
           "map_inds": torch.from_numpy(rng.integers(-1, 10000, Q))}
    bench.dump_outputs(out, str(tmp_path / "all"))
    for name, t in out.items():
        a = np.load(tmp_path / "all" / (name + ".npy"))
        assert a.dtype == np.float64 and np.array_equal(a, t.numpy()), name
    assert sorted(os.listdir(tmp_path / "all")) == sorted(n + ".npy" for n in out)
    # above the limit: the same seeded rows every time, their row numbers beside them, the whole dump within the limit
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 20 * 40)
    for d in ("a", "b"):
        bench.dump_outputs(out, str(tmp_path / d))
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == sorted([n + ".npy" for n in out] + ["sampled_quasars.npy"])
    rows = np.load(tmp_path / "a" / "sampled_quasars.npy").astype(np.int64)
    assert rows.size == 20 and np.all(np.diff(rows) > 0)
    assert sum(np.load(tmp_path / "a" / f).nbytes for f in files) <= 20 * 40
    for f in files:
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert np.array_equal(a, b), f
        if f != "sampled_quasars.npy":
            assert np.array_equal(a, out[f[:-4]].numpy()[rows]), f


@pytest.mark.gpu
def test_dump_outputs_are_the_timed_path_results(tmp_path):
    """The dumped arrays equal what DLAProcessor.process_device returns for the same seeded shard, and --steps sets the
    number of timed passes: the timed window holds `steps` times the launches of one pass."""
    import torch
    from gp_dla_detection_b200 import api, synthetic as syn
    Q, steps = 40, 3
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--quasars", str(Q), "--steps", str(steps),
                          "--warmup", "1", "--alt-steps", "0", "--strong-steps", "0", "--no-cpu-baseline",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900,
                         env=dict(os.environ, RANK="0", WORLD_SIZE="1", LOCAL_RANK="0"))
    assert res.returncode == 0, res.stderr[-2000:]
    d = json.loads(res.stdout)
    model = syn.make_model(20)
    proc = api.DLAProcessor(model, syn.make_samples(10000), syn.make_prior())
    try:
        pad = api.pad_spectra(syn.make_spectra(model, Q, shard=0))
        t = {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in pad.items()}
        n0 = proc.launch_count
        ref = proc.process_device(*[t[k] for k in ("wavelengths", "flux", "noise_variance", "pixel_mask", "lengths",
                                                   "z_qsos")])
        torch.cuda.synchronize()
        assert d["steps"] == steps and d["gpu_launches"] == steps * (proc.launch_count - n0)
    finally:
        proc.close()
    assert sorted(os.listdir(tmp_path)) == sorted(n + ".npy" for n in ref)
    for name, v in ref.items():
        a = np.load(tmp_path / (name + ".npy"))
        assert a.dtype == np.float64 and np.array_equal(a, v.cpu().numpy().astype(np.float64), equal_nan=True), name
