"""CPU: bench.py --dump-outputs writes float32 .npy files, whole when they fit the budget, else the same seeded sample
of points from every tensor, and stays under 64 MB at the benchmark's own output shapes."""
import os

import numpy as np
import torch

import bench


def _preds(n):
    # value = point index + 1e5 * channel: a dumped column tells which point it came from
    pts = torch.arange(n, dtype=torch.float32)
    return {name: (pts + 1e5 * torch.arange(c, dtype=torch.float32)[:, None]).expand(2, c, n).contiguous()
            for name, c in (("score", 3), ("frame_R", 9))}


def test_small_outputs_are_written_whole(tmp_path):
    preds = _preds(100)
    bench.dump_outputs(preds, str(tmp_path))
    for name, v in preds.items():
        got = np.load(tmp_path / (name + ".npy"))
        assert got.dtype == np.float32 and np.array_equal(got, v.numpy())


def test_large_outputs_share_one_fixed_sample(tmp_path):
    preds = _preds(1000)
    budget = 4 * 2 * 12 * 1000 // 5
    bench.dump_outputs(preds, str(tmp_path / "a"), budget=budget)
    bench.dump_outputs(preds, str(tmp_path / "b"), budget=budget)
    picked = []
    for name in preds:
        a, b = np.load(tmp_path / "a" / (name + ".npy")), np.load(tmp_path / "b" / (name + ".npy"))
        assert np.array_equal(a, b)
        picked.append(a[0, 0].astype(np.int64))
    assert sum(np.load(tmp_path / "a" / (n + ".npy")).nbytes for n in preds) <= budget
    assert np.array_equal(picked[0], picked[1]) and len(picked[0]) == 200
    assert np.all(np.diff(picked[0]) > 0)


def test_benchmark_sized_outputs_stay_under_64_mb(tmp_path):
    n = bench.NUM_POINTS
    preds = {name: torch.zeros(1).expand(64, c, n) for name, c in
             (("score", 3), ("frame_R", 9), ("frame_t", 4), ("movable_logits", 5))}
    bench.dump_outputs(preds, str(tmp_path))
    assert sum(os.path.getsize(tmp_path / f) for f in os.listdir(tmp_path)) <= 64 * 10 ** 6
