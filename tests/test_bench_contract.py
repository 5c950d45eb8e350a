"""bench.py contract on CPU: the reference arm (`--impl reference`) runs the CPU port of the path on a bounded sample
and prints ONE JSON line with the keys the driver reads; the GPU arm refuses to run without a B200 (no CPU fallback).
`--dump-outputs DIR` writes the predictions of the last timed step as DIR/<name>.npy."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from tests.helpers import ROOT


def test_reference_arm_prints_one_json_line(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "1", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "crystals/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["n_gpus"] == 1 and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["cores"] >= 1
    assert d["cpu_baseline"]["same_config"] is True and d["config"]["sample_crystals_per_step"] >= 64
    assert d["e2e"] == {"value": d["value"], "unit": "crystals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]
    assert "median of 1 steps after 1 warm-up" in d["cpu_baseline"]["sample"]
    assert os.listdir(tmp_path) == ["elastic_tensor_full.npy"]
    pred = np.load(tmp_path / "elastic_tensor_full.npy")
    assert pred.shape == (d["config"]["sample_crystals_per_step"], 6) and pred.dtype == np.float32
    assert np.isfinite(pred).all() and np.abs(pred).max() > 0


def test_gpu_arm_needs_a_gpu():
    import torch

    if torch.cuda.is_available():
        return
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "3"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode != 0 and "no CPU fallback" in out.stderr


@pytest.mark.gpu
def test_gpu_arm_dumps_the_predictions_of_the_last_step(tmp_path):
    """The dump holds what a caller of the timed forward receives: its first 64 crystals (the untiled unique ones) agree
    with the CPU oracle run with the same weights."""
    import torch

    import bench
    from matten_b200.model_factory import ScalarTensorModel
    from oracle import matten_restated as M
    from tests.helpers import rel_err, to_oracle_batch, tol

    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "3", "--no-train",
                          "--no-predict", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == 2
    assert os.listdir(tmp_path) == ["elastic_tensor_full.npy"]
    got = np.load(tmp_path / "elastic_tensor_full.npy")
    assert got.shape == (bench.CRYSTALS_PER_GPU, 6) and got.dtype == np.float32

    torch.manual_seed(0)  # bench.py's model
    prod = ScalarTensorModel(bench.HP, {"allowed_species": bench.SPECIES})
    orac = M.ScalarTensorModel(bench.HP, {"allowed_species": bench.SPECIES})
    orac.load_state_dict(prod.state_dict(), strict=False)
    with torch.no_grad():
        want = orac.eval()(to_oracle_batch(bench.make_batch(64, seed=0), torch.float32))
    assert rel_err(torch.from_numpy(got[:64]), want) < tol(torch.float32)
