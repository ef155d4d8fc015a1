"""bench.py's reference arm runs on the CPU: check the one-JSON-line contract and its keys here."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.nn as nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(*args):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                       timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = r.stdout.strip().splitlines()
    assert len(lines) == 1, lines
    return json.loads(lines[0])


def _dumped(path):
    arrays = {f[:-len(".npy")]: np.load(os.path.join(path, f)) for f in sorted(os.listdir(path))}
    assert all(f.endswith(".npy") for f in os.listdir(path))
    assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
    assert sum(a.nbytes for a in arrays.values()) <= 64_000_000
    return arrays


def test_reference_arm_dumps_the_last_step_and_repeats_it(tmp_path):
    """--steps K runs K timed steps; --dump-outputs writes the loss, forward outputs and gradients of the
    last one, and a second run with the same arguments writes the same arrays."""
    runs = []
    for i in range(2):
        d = _bench("--impl", "reference", "--workload", "fwfm", "--steps", "2", "--warmup", "1",
                   "--dump-outputs", str(tmp_path / f"run{i}"))
        assert d["steps"] == 2
        runs.append(_dumped(tmp_path / f"run{i}"))
    a, b = runs
    assert "loss" in a and "output_0" in a and any(k.startswith("grad.") for k in a)
    assert a.keys() == b.keys()
    for k in a:
        assert np.array_equal(a[k], b[k]), k


@pytest.mark.gpu
def test_cuda_arm_dumps_the_last_timed_step(tmp_path):
    d = _bench("--workload", "dcn", "--steps", "3", "--warmup", "1", "--no-others", "--no-aten", "--no-cpu-baseline",
               "--dump-outputs", str(tmp_path / "dump"))
    assert d["steps"] == 3
    arrays = _dumped(tmp_path / "dump")
    assert float(arrays["loss"]) == d["loss"]
    assert arrays["output_0"].shape == (d["config"]["batch_per_gpu"], 1)
    import rank_b200
    names = {k for k, _ in rank_b200.DCNModel(rank_b200.write_vocab_dir(str(tmp_path / "vocab")) + "/",
                                              hidden_units=[512, 256, 128], num_cross_layer=3).named_parameters()}
    assert {k for k in arrays if k.startswith("grad.")} == {"grad." + k for k in names}
    assert all(np.isfinite(a).all() for a in arrays.values())


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "fwfm",
                        "--steps", "1", "--warmup", "1"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = r.stdout.strip().splitlines()
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["impl"] == "reference" and d["unit"] == "samples/s" and d["higher_is_better"] is True
    assert d["config"]["workload"] and "model" not in d["config"]
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["value"] > 0 and d["warmup"] >= 3


def test_tower_runs_the_modules_on_cpu():
    """No CUDA tensor, no fused kernel: run_tower is exactly the reference's layer loop."""
    import rank_b200
    from rank_b200 import tower
    torch.manual_seed(0)
    layers = nn.ModuleList([nn.Linear(6, 8), rank_b200.Dice(8), nn.BatchNorm1d(8), nn.Linear(8, 4), nn.BatchNorm1d(4),
                            nn.ReLU(), nn.Linear(4, 1)]).train()
    x = torch.randn(512, 6)
    a = tower.run_tower(layers, x)
    torch.manual_seed(0)
    b = x
    for m in layers:
        b = m(b)
    # the second pass updated the running statistics again, the outputs of a training-mode pass do not depend on them
    assert torch.equal(a, b)
