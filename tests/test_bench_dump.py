"""bench.py --dump-outputs: what the last timed step computed, written so that two builds can be
compared output for output."""
import os
import subprocess
import sys

import numpy as np
import pytest

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class _Results:
    """The two read-backs step_outputs takes from a BatchedArena, on the host."""

    def __init__(self, n):
        import torch
        self.n_envs = n
        self._out = torch.arange(n * 8, dtype=torch.int32).view(n, 8) - 5
        self._hash = torch.from_numpy(np.arange(n, dtype=np.uint64) * np.uint64(0x9E3779B97F4A7C15)).view(torch.int64)

    def step_out(self):
        return self._out

    def state_hash(self):
        return self._hash


@pytest.mark.parametrize("n", [7, 1 << 20])
def test_step_outputs_are_exact_and_bounded(n):
    d = bench.step_outputs(_Results(n))
    assert all(a.dtype == np.float64 for a in d.values())
    assert sum(a.nbytes for a in d.values()) <= bench.DUMP_LIMIT
    ids = d["env_ids"].astype(np.int64)
    assert len(ids) == (n if n * 88 <= bench.DUMP_LIMIT else bench.DUMP_LIMIT // 88)
    assert (np.diff(ids) > 0).all() and (bench.step_outputs(_Results(n))["env_ids"] == d["env_ids"]).all()
    assert (d["step_out"] == np.arange(n * 8).reshape(n, 8)[ids] - 5).all()
    lo, hi = d["state_hash_lo_hi"].astype(np.uint64).T
    assert (lo | (hi << np.uint64(32)) == ids.astype(np.uint64) * np.uint64(0x9E3779B97F4A7C15)).all()


@pytest.mark.gpu
def test_dump_repeats_and_follows_the_step_count(tmp_path):
    def run(steps, name):
        out = tmp_path / name
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--envs", "512", "--prewarm", "64",
                            "--steps", str(steps), "--warmup", "1", "--no-cpu", "--no-obs", "--dump-outputs", str(out)],
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-4000:]
        return {f[:-4]: np.load(out / f) for f in sorted(os.listdir(out))}

    a, b, c = run(4, "a"), run(4, "b"), run(3, "c")
    assert sorted(a) == ["env_ids", "state_hash_lo_hi", "step_out"]
    assert a["step_out"].shape == (512, 8) and a["state_hash_lo_hi"].shape == (512, 2)
    assert all(np.array_equal(a[k], b[k]) for k in a), "the same arguments gave different outputs"
    assert not np.array_equal(a["state_hash_lo_hi"], c["state_hash_lo_hi"]), "--steps did not change the timed steps"
