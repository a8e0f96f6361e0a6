"""CPU: `bench.py --dump-outputs DIR` writes a fixed, seeded float64 sample of what the timed step
computed, within 64 MB, and refuses the arguments it cannot honour."""
import os
import sys

import numpy as np
import pytest

import bench


class _Batch:
    """Stands in for eggshell_b200.Batch: every body of world k sits at p = k."""

    def __init__(self, W, n):
        self.W, self.n = W, n

    def bodies(self):
        k = np.arange(self.W, dtype=np.float64)[:, None, None]
        return (np.broadcast_to(k, (self.W, self.n, 3)), np.broadcast_to(k[..., None], (self.W, self.n, 3, 3)),
                np.broadcast_to(-k, (self.W, self.n, 3)), np.broadcast_to(2 * k, (self.W, self.n, 3)))


def _dump(path, W, n):
    st = {"sweeps": np.arange(W, dtype=np.int32), "residual": np.arange(W, dtype=np.float64)}
    bench.dump_outputs(str(path), _Batch(W, n), st, np.arange(W, dtype=np.float64))
    return {f[:-4]: np.load(os.path.join(path, f)) for f in os.listdir(path)}


def test_dump_is_a_fixed_float64_sample_within_64_mb(tmp_path):
    W, n = 65536, 64                                   # the c3 batch
    a, b = _dump(tmp_path / "a", W, n), _dump(tmp_path / "b", W, n)
    assert set(a) == {"p", "R", "v", "w", "sweeps", "residual", "cost"}
    assert all(x.dtype == np.float64 for x in a.values())
    assert sum(x.nbytes for x in a.values()) <= 64 << 20
    idx = a["p"][:, 0, 0]
    assert len(idx) == bench.DUMP_WORLDS and np.all(np.diff(idx) > 0) and idx[-1] < W
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    assert np.array_equal(a["sweeps"], idx) and np.array_equal(a["cost"], idx) and np.array_equal(a["v"][:, 0, 0], -idx)


def test_dump_keeps_every_world_of_a_small_batch(tmp_path):
    out = _dump(tmp_path, 7, 32)
    assert np.array_equal(out["p"][:, 0, 0], np.arange(7)) and out["R"].shape == (7, 32, 3, 3)


@pytest.mark.parametrize("argv", [["--impl", "reference", "--dump-outputs", "d"], ["--steps", "0", "--dump-outputs", "d"]])
def test_dump_refuses_arguments_without_a_timed_gpu_step(argv, monkeypatch):
    monkeypatch.setattr(sys, "argv", ["bench.py"] + argv)
    with pytest.raises(SystemExit):
        bench.parse()
