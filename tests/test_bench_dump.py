"""bench.py --dump-outputs: the timed path's last output lands in DIR/<name>.npy (float32, at most 64 MB in all, a fixed seeded
sample when larger), so that two builds can be compared output for output on identical inputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(*args):
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE")}
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-800:]
    return json.loads(r.stdout.strip().splitlines()[-1])


def test_dump_samples_large_outputs_with_a_fixed_seed(tmp_path):
    import bench
    big = torch.arange(bench.DUMP_BYTES // 4 + 1000, dtype=torch.float32).view(-1, 8)
    small = torch.ones(3, dtype=torch.float16)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"big": big, "small": small})
    a, b = np.load(tmp_path / "a" / "big.npy"), np.load(tmp_path / "b" / "big.npy")
    assert a.dtype == np.float32 and a.nbytes == bench.DUMP_BYTES // 2 and np.array_equal(a, b)
    assert np.all(np.diff(a) > 0)                                    # distinct elements of the flattened array, in order
    s = np.load(tmp_path / "a" / "small.npy")
    assert s.dtype == np.float32 and np.array_equal(s, np.ones(3, np.float32))
    assert sum(os.path.getsize(p) for p in (tmp_path / "a").iterdir()) <= 64 << 20


def test_reference_arm_dumps_its_last_step(tmp_path):
    d = _bench("--impl", "reference", "--workload", "cfg1_tiny", "--steps", "2", "--warmup", "1", "--dump-outputs", str(tmp_path))
    assert d["steps"] == 2
    bev = np.load(tmp_path / "bev.npy")
    assert bev.dtype == np.float32 and bev.shape == (1, 64, 50, 50) and np.abs(bev).max() > 0


@pytest.mark.gpu
def test_timed_path_dump_is_the_lift_of_the_bench_inputs(tmp_path):
    """The flagship path (graph replay of the forward lift) at a size that is stored whole, against the oracle's fp64 lift of the
    inputs bench.py builds for rank 0 (seed 100)."""
    from fiery_b200.synthetic import CONFIGS, make_calibration, make_head
    from oracle import lift_oracle as O
    d = _bench("--workload", "cfg1_tiny", "--steps", "3", "--warmup", "1", "--no-cpu-baseline", "--no-extras",
               "--dump-outputs", str(tmp_path))
    assert d["steps"] == 3
    cfg = CONFIGS["cfg1_tiny"]
    K, E = (torch.from_numpy(a) for a in make_calibration(cfg, seed=100))
    exact = O.LiftOracle.from_config(cfg).lift_exact(torch.from_numpy(make_head(cfg, seed=100)), K, E)
    bev = np.load(tmp_path / "bev.npy")
    assert bev.dtype == np.float32 and bev.shape == tuple(exact.shape)
    assert O.normwise_error(torch.from_numpy(bev), exact) < 1e-4
