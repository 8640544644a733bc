"""CPU: the reference arm of bench.py runs without a GPU and prints one JSON line with the contract's keys."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--roots", "16", "--sims", "4",
                          "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in line, k
    assert line["impl"] == "reference" and line["value"] > 0 and line["vs_baseline"] is None
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0


def test_reference_arm_non_zero_ranks_exit_silently():
    """Under torchrun (N > 1) rank 0 alone runs the reference arm; the other ranks exit 0 without work or output."""
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT="29555")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                          "--warmup", "0"], capture_output=True, text=True, timeout=120, env=env)
    assert out.returncode == 0 and out.stdout.strip() == "", out.stderr[-1000:]


def test_dump_outputs_float32_and_fixed_root_sample_above_the_limit(tmp_path):
    import torch

    import bench

    B = 100
    out = {"value": torch.arange(B, dtype=torch.float32) / 7, "visit_count": torch.arange(B * 10, dtype=torch.int32).view(B, 10)}
    bench.dump_outputs(str(tmp_path / "all"), out)
    assert sorted(os.listdir(tmp_path / "all")) == ["value.npy", "visit_count.npy"]
    v = np.load(tmp_path / "all" / "visit_count.npy")
    assert v.dtype == np.float32 and np.array_equal(v, out["visit_count"].numpy())

    limit = 4096                                        # 100 roots x 44 bytes do not fit: a sample of roots is written
    for d in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / d), out, limit=limit)
        files = [tmp_path / d / f for f in os.listdir(tmp_path / d)]
        assert sum(os.path.getsize(f) for f in files) <= limit
    idx = np.load(tmp_path / "s1" / "root_index.npy")
    assert idx.dtype == np.float64 and 0 < len(idx) < B and (np.diff(idx) > 0).all()
    assert np.array_equal(idx, np.load(tmp_path / "s2" / "root_index.npy"))
    k = idx.astype(np.int64)
    assert np.array_equal(np.load(tmp_path / "s1" / "value.npy"), out["value"].numpy()[k])
    assert np.array_equal(np.load(tmp_path / "s1" / "visit_count.npy"), out["visit_count"].numpy()[k].astype(np.float32))


def test_steps_below_one_rejected():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True, timeout=120)
    assert out.returncode == 2 and "--steps" in out.stderr
