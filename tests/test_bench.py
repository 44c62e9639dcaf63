"""bench.py --dump-outputs: what the timed step computed, written where two builds can compare it."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def test_dump_outputs_samples_large_buffers_the_same_way_every_time(tmp_path):
    n = 10_000_000  # float32 holds every index exactly: a sampled value is its own position
    tensors = [torch.arange(n, dtype=torch.float32), -torch.arange(n, dtype=torch.float32)]
    bench.dump_outputs(str(tmp_path / "a"), tensors, rank=0, world=1)
    bench.dump_outputs(str(tmp_path / "b"), tensors, rank=0, world=1)
    total = 0
    for i in range(2):
        a = np.load(tmp_path / "a" / f"rank0_buffer{i}.npy")
        b = np.load(tmp_path / "b" / f"rank0_buffer{i}.npy")
        total += os.path.getsize(tmp_path / "a" / f"rank0_buffer{i}.npy")
        assert a.dtype == np.float32 and np.array_equal(a, b)
        pos = -a if i else a
        assert 0 < len(pos) <= bench.DUMP_BYTES // 4 // 2
        assert np.all(np.diff(pos) > 0) and pos[0] >= 0 and pos[-1] < n
    assert total <= 64 << 20


def test_dump_outputs_keeps_small_buffers_whole(tmp_path):
    t = torch.linspace(-1, 1, 1000, dtype=torch.float64)
    bench.dump_outputs(str(tmp_path), [t], rank=3, world=4)
    got = np.load(tmp_path / "rank3_buffer0.npy")
    assert got.dtype == np.float32 and np.array_equal(got, t.float().numpy())


@pytest.mark.gpu
def test_bench_dumps_the_last_timed_step(tmp_path):
    """At N=1 a step sums the two buffers into both: with inputs i + 2j, the first step gives
    1 + 4j and every further step doubles it. One check run, W warmup and K timed steps leave
    (1 + 4j) * 2^(W + K)."""
    steps, warmup, n = 2, 3, 3_000_000
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps),
                          "--warmup", str(warmup), "--elements", str(n), "--no-sweep", "--dump-outputs", str(tmp_path)],
                         env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-3000:]
    res = json.loads(out.stdout.strip().splitlines()[-1])
    assert res["steps"] == steps and res["gpu_launches"] == steps
    want = (1 + 4 * np.arange(n, dtype=np.float64)) * 2.0 ** (warmup + steps)
    for i in range(2):
        got = np.load(tmp_path / f"rank0_buffer{i}.npy")
        assert got.dtype == np.float32 and np.array_equal(got.astype(np.float64), want)
