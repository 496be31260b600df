"""CPU: bench.py's host-side helpers (config block, ncu-summary lookup, reference arm on a tiny sample)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from tests import util

sys.path.insert(0, util.ROOT)
import bench  # noqa: E402


def test_workload_config_is_identical_for_both_arms():
    a = bench.workload_config(64, 1, 64, 64)
    b = bench.workload_config(64, 1, 64, 64)
    assert a == b and a["v2v_chunk_frames"] == 64 and a["volume_size"] == 64 and "configs[1]" in a["workload"]
    assert "configs[3]" in bench.workload_config(8, 1, 128, 8)["workload"]
    big = bench.workload_config(1024, 1, 64, 64, strong=True, features=False)
    assert "NOT materialised" in big["outputs"]


def test_ncu_traffic_lookup_matches_launch_size():
    hit = bench.ncu_traffic("conv_march_kernel<2, 0, 2, 1>", 64, 64)
    assert hit is not None and hit[1].startswith("profiles/") and hit[0]["frames_per_launch"] == 64
    total = hit[0]["dram_bytes_read"] + hit[0]["dram_bytes_write"]
    assert 2.0e9 < total < 2.5e9                       # 2.15 GB algorithmic at 64 frames per launch
    assert bench.ncu_traffic("conv_march_kernel<2, 0, 2, 1>", 16, 64) is None      # no capture at that launch size: null
    assert bench.ncu_traffic("conv_march_kernel<2, 0, 2, 1>", 64, 128) is None


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    """`bench.py --impl reference` (the oracle port on the host cores) on the smallest sample: one JSON line, the keys the
    driver reads, the real per-step sample stated (1 frame per step)."""
    r = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--steps", "1", "--warmup", "0"], cwd=util.ROOT,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-1500:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["frames_run_per_step"] == 1 and d["cpu_baseline"]["kind"] == "port"
    assert d["config"] == bench.workload_config(64, 1, 64, 64) and d["value"] > 0 and d["e2e"]["h2d_bytes_per_step"] == 0


def test_dump_outputs_writes_float32_and_a_fixed_sample(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_SAMPLE", 100)
    kp = torch.randn(2, 15, 3)
    big = torch.arange(1000, dtype=torch.float64).reshape(10, 100)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"keypoints_3d": kp, "features": None, "volumes": big})
    assert sorted(os.listdir(tmp_path / "a")) == ["keypoints_3d.npy", "volumes.npy"]
    k = np.load(tmp_path / "a" / "keypoints_3d.npy")
    assert k.dtype == np.float32 and np.array_equal(k, kp.numpy())             # small outputs: whole, shape kept
    va, vb = np.load(tmp_path / "a" / "volumes.npy"), np.load(tmp_path / "b" / "volumes.npy")
    assert va.dtype == np.float32 and va.shape == (100,) and np.array_equal(va, vb)
    assert np.all(np.diff(va) >= 0) and len(np.unique(va)) > 50                # ascending flat indices, spread out


@pytest.mark.gpu
def test_bench_dumps_the_same_outputs_from_run_to_run(tmp_path):
    """`bench.py --dump-outputs` twice with the same arguments: the last timed step's outputs agree bit for bit."""
    for d in ("a", "b"):
        r = subprocess.run([sys.executable, "bench.py", "--steps", "2", "--warmup", "0", "--frames-per-gpu", "2",
                            "--no-kernel-table", "--no-cpu-baseline", "--dump-outputs", str(tmp_path / d)],
                           cwd=util.ROOT, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-1500:]
        line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
        assert line["steps"] == 2
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == ["coord_volumes.npy", "features.npy", "keypoints_3d.npy", "volumes.npy"]
    total = 0
    for n in names:
        a, b = np.load(tmp_path / "a" / n), np.load(tmp_path / "b" / n)
        assert a.dtype == np.float32 and np.array_equal(a, b), n
        total += a.nbytes
    assert total <= 64 << 20
    kp = np.load(tmp_path / "a" / "keypoints_3d.npy")
    assert kp.shape == (2, 15, 3) and np.isfinite(kp).all()
