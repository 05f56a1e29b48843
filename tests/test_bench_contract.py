"""bench.py host logic (CPU): the workloads are BASELINE.json's configurations, the algorithmic-byte model is the one
SURVEY.md section 8(d) states, the synthetic batches have the reference datasets' padding, and the `--impl reference` arm
prints the contract line around the vendored reference (or the oracle port when baseline/_ref is absent)."""
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_workloads_are_the_baseline_configurations():
    cfgs = json.load(open(os.path.join(ROOT, "BASELINE.json")))["configs"]
    want = {"h36m": cfgs[0], "cmu": cfgs[1], "3dpw": cfgs[2], "stress": cfgs[4]}
    for name, text in want.items():
        layout, v, t_in, t_out, _ = bench.WORKLOADS[name]
        m = re.search(r"(\d+) joints", text)
        joints = int(m.group(1)) if m else 22        # "H3.6M joints" (stress) = 22
        frames = re.search(r"(\d+)\D+(\d+) frames", text)
        assert v == joints, name
        assert (t_in, t_out) == (int(frames.group(1)), int(frames.group(2))), name
    assert bench.feat("stress") == 256 and bench.feat("h36m") == 64          # "256 hidden channels"
    assert bench.DEFAULT_BATCH.get("stress") == 32


def test_algorithmic_bytes_follow_survey_8d():
    # one HBM round trip per DSTDGCB layer, fp32: fwd 4 T V sum(Cin + Cout), bwd 4 T V sum(2 Cin + Cout)
    t, v, c = 35, 22, 64
    chans = [(6, c)] + [(c, c)] * 5 + [(c, 3)]
    fwd = 4 * t * v * sum(a + b for a, b in chans)
    bwd = 4 * t * v * sum(2 * a + b for a, b in chans)
    assert bench.algorithmic_bytes_per_pass(v, t) == fwd + bwd == 5_987_520
    assert bench.algorithmic_bytes_per_pass(22, 125, 256) == 84_744_000      # the stress line's scope string


def test_synthetic_batch_has_the_dataset_padding():
    n, t, v, t_in = 3, 35, 22, 10
    x, x_inv, seq = bench.synthetic_batch(n, t, v, t_in, seed=5)
    assert x.shape == x_inv.shape == seq.shape == (n, t, 3 * v)
    assert torch.equal(x[:, :t_in], seq[:, :t_in])                            # observed frames
    assert torch.equal(x[:, t_in:], seq[:, t_in - 1:t_in].expand(-1, t - t_in, -1))   # last observed frame repeated
    rev = torch.flip(seq, dims=[1])
    assert torch.equal(x_inv[:, :t_in], rev[:, :t_in])
    assert torch.equal(x_inv[:, t_in:], rev[:, t_in - 1:t_in].expand(-1, t - t_in, -1))
    x2, _, _ = bench.synthetic_batch(n, t, v, t_in, seed=5)
    assert torch.equal(x, x2)                                                 # seeded


def test_workload_config_names_the_workload():
    class A:
        workload, batch, gpus = "3dpw", 64, 4
    cfg = bench.workload_config(A)
    assert "3dpw" in cfg["workload"] and "23 joints" in cfg["workload"] and "10->30" in cfg["workload"]
    assert cfg["batch_per_gpu"] == 64 and cfg["global_batch"] == 256 and cfg["inverse"] is True and cfg["dropout"] == 0.0
    assert "model" not in cfg


def test_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference`: one JSON line with impl / metric / unit / cpu_baseline / e2e (zero copy bytes), timed on
    the host cores; tiny batch so that it runs in seconds."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--batch", "4", "--steps", "2",
                        "--warmup", "1", "--cpu-seconds", "0"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "train_samples_per_s" and line["unit"] == "samples/s"
    assert line["higher_is_better"] is True and line["value"] > 0 and line["steps"] == 2 and line["warmup"] >= 1
    cb = line["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == line["value"]
    if os.path.exists(os.path.join(ROOT, "baseline", "_ref", "engine", "prediction.py")):
        assert cb["kind"] == "reference"                                      # the unmodified reference, not the port
    assert line["e2e"] == {"value": line["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["config"]["batch_per_gpu"] == 4 and "h36m" in line["config"]["workload"]


def test_dump_outputs_samples_large_arrays_within_the_limit(tmp_path):
    """Small arrays are written whole, larger ones as the same seeded sample every time, all within the byte limit."""
    rng = np.random.default_rng(1)
    arrays = {"small": rng.standard_normal(10).astype(np.float32), "count": np.array(7, dtype=np.int64),
              "wide": rng.standard_normal((300, 300)).astype(np.float32), "big": rng.standard_normal(100_000)}
    limit = 256 << 10
    for run in ("a", "b"):
        assert bench.dump_outputs(str(tmp_path / run), arrays, limit=limit) <= limit
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["big.npy", "count.npy", "small.npy", "wide.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= limit
    got = {n: np.load(tmp_path / "a" / f"{n}.npy") for n in arrays}
    assert got["small"].dtype == np.float32 and np.array_equal(got["small"], arrays["small"])
    assert got["count"].dtype == np.float64 and got["count"] == 7
    assert got["big"].dtype == np.float64 and got["wide"].dtype == np.float32
    for n in ("big", "wide"):
        assert 0 < got[n].size < arrays[n].size and np.isin(got[n], arrays[n]).all()
    for n in arrays:
        assert np.array_equal(got[n], np.load(tmp_path / "b" / f"{n}.npy"))


def test_steps_must_be_positive():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True,
                       timeout=120, cwd=ROOT)
    assert r.returncode == 2 and "--steps" in r.stderr


@pytest.mark.gpu
def test_dump_outputs_are_identical_from_run_to_run(tmp_path):
    """`bench.py --dump-outputs`: the loss, model state and gradients of the last timed step, float32 / float64 files
    within 64 MB, bit-identical for two runs with the same arguments (seeded inputs and weights, deterministic kernels)."""
    dumps = []
    for run in range(2):
        out = tmp_path / f"run{run}"
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--batch", "8", "--steps", "3",
                            "--warmup", "3", "--no-secondary", "--no-cpu-baseline", "--no-gpu-eager-baseline",
                            "--dump-outputs", str(out)], capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 3
        files = sorted(os.listdir(out))
        assert sum(os.path.getsize(out / f) for f in files) <= bench.DUMP_LIMIT
        dumps.append({f: np.load(out / f) for f in files})
    a, b = dumps
    assert a.keys() == b.keys() and "loss.npy" in a and np.isfinite(a["loss.npy"]).all()
    assert "state.encoders.0.0.stgcn.0.0.W_s.npy" in a and "grad.encoders.0.0.stgcn.0.0.W_s.npy" in a
    for f in a:
        assert a[f].dtype in (np.float32, np.float64), f
        assert np.array_equal(a[f], b[f]), f
