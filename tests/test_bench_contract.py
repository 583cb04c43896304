"""bench.py's reference arm runs without a GPU: one JSON line with the contract's keys. On a GPU: --dump-outputs."""

import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert res.returncode == 0, res.stderr
    lines = [l for l in res.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "Mpx/s disparity" and d["unit"] == "Mpx/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1
    assert d["value"] > 0 and d["cpu_baseline"]["value"] == d["value"] and d["cpu_baseline"]["kind"] in ("reference", "port")
    assert d["cpu_baseline"]["cores"] >= 1 and "rows" in d["cpu_baseline"]["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "Mpx/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert res.returncode == 0 and res.stdout.strip() == ""


@pytest.mark.gpu
def test_dump_outputs_are_finite_and_repeatable(tmp_path):
    """--dump-outputs: the timed path's last-step outputs as finite float32 arrays (NaN cells as 0 beside validity
    masks), within 64 MB, and the same files from two runs with the same arguments."""
    import numpy as np
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    dumps = []
    for run in ("a", "b"):
        res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1",
                              "--no-cpu-baseline", "--dump-outputs", str(tmp_path / run)],
                             capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert res.returncode == 0, res.stderr
        assert json.loads(res.stdout.strip().splitlines()[-1])["steps"] == 1
        dumps.append({p.name: np.load(p) for p in sorted((tmp_path / run).iterdir())})
    a, b = dumps
    names = {f"{kind}{suffix}_{f}.npy" for kind in ("disparity", "corrmap") for suffix in ("", "_valid") for f in range(4)}
    assert set(a) == names and set(b) == names
    assert sum(x.nbytes for x in a.values()) <= 64 << 20
    for name, x in a.items():
        assert x.dtype == np.float32 and x.shape == (384, 2048) and np.isfinite(x).all(), name
        assert np.array_equal(x, b[name]), name
        if "_valid_" in name:
            assert set(np.unique(x)) <= {0.0, 1.0} and x.mean() > 0.5, name
            assert (a[name.replace("_valid", "")][x == 0] == 0).all(), name
