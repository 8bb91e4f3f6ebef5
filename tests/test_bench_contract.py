"""CPU: the reference arm of bench.py (`--impl reference`: the oracle port timed on the host cores) prints one JSON line with the
keys the measurement contract names; the effective host thread count honours affinity and the cgroup quota; --dump-outputs
writes float32 arrays within its size limit (GPU: the poses of our arm's last timed step)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "impl", "cpu_baseline", "e2e"):
        assert k in line, k
    assert line["impl"] == "reference" and line["metric"] == "poses/sec" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert line["config"]["workload"] == "pem_matching_32x2048x2048"


def _bench_module():
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    return b


def test_host_threads_is_bounded_by_affinity():
    b = _bench_module()
    n = b.host_threads()
    assert 1 <= n <= (os.cpu_count() or 1)
    assert n <= len(os.sched_getaffinity(0))


def test_dump_outputs_writes_float32_and_one_fixed_sample_above_the_limit(tmp_path):
    import numpy as np
    import torch
    b = _bench_module()
    g = torch.Generator().manual_seed(0)
    arrays = dict(pred_R=torch.randn(100, 3, 3, generator=g, dtype=torch.float64), pred_t=torch.randn(100, 3, generator=g),
                  pred_pose_score=torch.rand(100, generator=g))
    b.dump_outputs(str(tmp_path / "all"), arrays)
    for k, v in arrays.items():
        got = np.load(tmp_path / "all" / (k + ".npy"))
        assert got.dtype == np.float32 and np.array_equal(got, v.float().numpy())
    per_row = 4 * (9 + 3 + 1)
    for run in ("a", "b"):
        b.dump_outputs(str(tmp_path / run), arrays, limit_bytes=30 * per_row + 5)
    got = {k: np.load(tmp_path / "a" / (k + ".npy")) for k in arrays}
    assert all(v.shape[0] == 30 for v in got.values())
    assert sum(v.nbytes for v in got.values()) <= 30 * per_row + 5
    rows = [int(np.flatnonzero((arrays["pred_t"].numpy() == r).all(axis=1))[0]) for r in got["pred_t"]]
    assert rows == sorted(rows) and len(set(rows)) == 30
    for k, v in arrays.items():                                   # the same proposals in every array and in every run
        assert np.array_equal(got[k], v.float().numpy()[rows])
        assert np.array_equal(got[k], np.load(tmp_path / "b" / (k + ".npy")))


@pytest.mark.gpu
def test_ours_dumps_the_poses_of_its_last_timed_step(tmp_path):
    import numpy as np
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--no-cpu-baseline",
                          "--no-ref-gpu", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2
    B = line["config"]["proposals_per_gpu"]
    shapes = dict(init_R=(B, 3, 3), init_t=(B, 3), pred_R=(B, 3, 3), pred_t=(B, 3), pred_pose_score=(B,))
    assert sorted(os.listdir(tmp_path)) == sorted(k + ".npy" for k in shapes)
    got = {k: np.load(tmp_path / (k + ".npy")) for k in shapes}
    for k, shape in shapes.items():
        assert got[k].dtype == np.float32 and got[k].shape == shape and np.isfinite(got[k]).all(), k
    R = got["pred_R"].astype(np.float64)
    assert np.abs(R @ R.transpose(0, 2, 1) - np.eye(3)).max() < 1e-4
