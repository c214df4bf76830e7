"""bench.py --dump-outputs: what the last timed step computed, written so two builds can be compared array for array."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_writes_the_loss_and_a_fixed_sample_of_the_parameters(tmp_path, monkeypatch):
    import bench
    torch.manual_seed(0)
    model = torch.nn.Sequential(torch.nn.Linear(30, 20), torch.nn.BatchNorm1d(20))
    flat = torch.cat([p.detach().reshape(-1) for p in model.parameters()]).numpy()
    bench.dump_outputs(str(tmp_path / "whole"), torch.tensor(0.25), model)
    assert sorted(os.listdir(tmp_path / "whole")) == ["loss.npy", "params.npy"]
    assert np.load(tmp_path / "whole" / "loss.npy").tolist() == [0.25]
    whole = np.load(tmp_path / "whole" / "params.npy")
    assert whole.dtype == np.float32 and np.array_equal(whole, flat)
    monkeypatch.setattr(bench, "DUMP_SAMPLE", 100)                 # 660 parameters: a sample, at the same positions every time
    bench.dump_outputs(str(tmp_path / "a"), torch.tensor(0.25), model)
    bench.dump_outputs(str(tmp_path / "b"), torch.tensor(0.25), model)
    a, b = np.load(tmp_path / "a" / "params.npy"), np.load(tmp_path / "b" / "params.npy")
    assert a.shape == (100,) and np.array_equal(a, b) and np.isin(a, flat).all()


@pytest.mark.gpu
def test_bench_dump_is_reproducible(tmp_path):
    """Two runs with the same arguments time exactly --steps steps and leave the same outputs (same inputs, same seeds)."""
    runs = []
    for name in ("a", "b"):
        res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--model", "foo", "--gpus", "1", "--steps", "3",
                              "--warmup", "5", "--dump-outputs", str(tmp_path / name)],
                             capture_output=True, text=True, timeout=600, cwd=str(tmp_path))
        assert res.returncode == 0, res.stderr[-3000:]
        out = json.loads([line for line in res.stdout.splitlines() if line.startswith("{")][-1])
        assert out["steps"] == 3
        runs.append(tmp_path / name)
    for n in ("loss.npy", "params.npy"):
        a, b = np.load(runs[0] / n), np.load(runs[1] / n)
        assert a.dtype == np.float32 and np.allclose(a, b, rtol=1e-5, atol=1e-6), n
