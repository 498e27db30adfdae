"""bench.py --dump-outputs: float32 .npy files, large arrays reduced to the same seeded sample in every run, and
the whole dump kept under 64 MB (no GPU needed for the writer itself)."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_is_float32_sampled_and_repeatable(tmp_path):
    g = torch.Generator().manual_seed(0)
    big = torch.arange(3 * bench.DUMP_MAX_ELEMENTS, dtype=torch.float32).view(3, -1)     # value = flat position
    arrays = [("loss", torch.tensor(2.5, dtype=torch.float64)), ("logits", torch.randn(4, 5, generator=g).half()),
              ("grad.w", big)]
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    assert sorted(os.listdir(tmp_path / "a")) == ["grad.w.npy", "logits.npy", "loss.npy"]
    for name in os.listdir(tmp_path / "a"):
        a, b = np.load(tmp_path / "a" / name), np.load(tmp_path / "b" / name)
        assert a.dtype == np.float32 and np.array_equal(a, b), name
    assert np.load(tmp_path / "a" / "loss.npy") == np.float32(2.5)
    assert np.array_equal(np.load(tmp_path / "a" / "logits.npy"), arrays[1][1].float().numpy())
    w = np.load(tmp_path / "a" / "grad.w.npy")
    assert w.shape == (bench.DUMP_MAX_ELEMENTS,)
    assert (np.diff(w) > 0).all() and w[0] >= 0 and w[-1] < big.numel()         # distinct positions, in order


def test_dump_refuses_more_than_64_mb(tmp_path):
    n = int(64e6) // (4 * bench.DUMP_MAX_ELEMENTS) + 1
    arrays = [("grad.%d" % i, torch.zeros(bench.DUMP_MAX_ELEMENTS)) for i in range(n)]
    with pytest.raises(AssertionError, match="64 MB"):
        bench.dump_outputs(str(tmp_path), arrays)


@pytest.mark.parametrize("flags", [["--steps", "0"], ["--warmup", "-1"]])
def test_bench_rejects_step_counts_it_cannot_run(flags):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + flags, capture_output=True, text=True)
    assert r.returncode == 2 and "--steps must be >= 1" in r.stderr
