"""world_size-2 CPU (gloo) test of the N>1 host path: contiguous world shards + the cost allgather
+ identical selection on every rank (SURVEY.md §8e)."""
import numpy as np
import torch

from eggshell_b200 import mpc
from tests.mpc_helpers import run_ranks


def test_shard_range_partitions_exactly():
    for total in (1, 7, 64, 65536, 1048576 + 3):
        for ws in (1, 2, 3, 8):
            spans = [mpc.shard_range(total, r, ws) for r in range(ws)]
            assert spans[0][0] == 0 and spans[-1][1] == total
            assert all(spans[i][1] == spans[i + 1][0] for i in range(ws - 1))
            sizes = [hi - lo for lo, hi in spans]
            assert max(sizes) - min(sizes) <= 1
            for g in (0, total // 2, total - 1):
                r, l = mpc.owner_of(g, total, ws)
                assert spans[r][0] + l == g


def _worker(rank, ws, total):
    lo, hi = mpc.shard_range(total, rank, ws)
    # deterministic per-world "rollout cost" that depends only on the global world index
    g = np.arange(lo, hi, dtype=np.float64)
    local = torch.from_numpy(np.cos(g * 0.37) + 1e-3 * g)
    allc = mpc.allgather_costs(local)
    idx, val = mpc.select_best(allc, k=3)
    return allc.numpy().copy(), idx.copy(), val.copy()


def _run(total):
    res = run_ranks(_worker, 2, "gloo", total, timeout=120)
    g = np.arange(total, dtype=np.float64)
    expect = np.cos(g * 0.37) + 1e-3 * g
    for allc, idx, val in res:
        assert np.array_equal(allc, expect)
        assert np.array_equal(idx, np.argsort(expect, kind="stable")[:3])
    assert np.array_equal(res[0][1], res[1][1])


def test_allgather_even_shards_gloo():
    _run(64)


def test_allgather_uneven_shards_gloo():
    _run(37)
