"""Host-side id handling of the mutable index (no GPU): validation of ids against one index, and the per-rank
filtering of a global id list over the shards of ShardedIndex.shard_bounds."""
import numpy as np
import pytest
import torch

from mdir_b200 import MdirError
from mdir_b200.search import ShardedIndex, check_ids, ids_for_rank


def test_check_ids_maps_to_rows_and_rejects_outside():
    assert np.array_equal(check_ids([1000, 1005, 1005, 1099], 1000, 1100), [0, 5, 5, 99])
    assert np.array_equal(check_ids(torch.tensor([7, 3]), 0, 8), [7, 3])
    assert np.array_equal(check_ids(np.array([[2, 3]], dtype=np.int32), 2, 4), [0, 1])
    assert check_ids([], 0, 10).shape == (0,)
    for bad in ([999], [1100], [1000, -1], [2 ** 40]):
        with pytest.raises(MdirError):
            check_ids(bad, 1000, 1100)
    with pytest.raises(MdirError):
        check_ids([1.5], 0, 10)


@pytest.mark.parametrize("n_total,world", [(10, 3), (60013, 4), (7, 8), (1001001, 8)])
def test_ids_for_rank_partitions_a_global_list(n_total, world):
    ranges = [ShardedIndex.shard_bounds(n_total, world, r) for r in range(world)]
    rs = np.random.RandomState(n_total)
    ids = rs.randint(0, n_total, 500)
    ids = np.concatenate([ids, ids[:50], [0, n_total - 1]])
    parts = [ids_for_rank(ids, ranges, r) for r in range(world)]
    assert sum(len(p) for p in parts) == len(ids)                    # every id lands on exactly one rank
    for r, p in enumerate(parts):
        lo, hi = ranges[r]
        assert ((p >= lo) & (p < hi)).all()
        assert np.array_equal(p, ids[(ids >= lo) & (ids < hi)])      # order and repeats kept
    for bad in ([n_total], [-1], [0, n_total + 7]):
        with pytest.raises(MdirError):
            ids_for_rank(bad, ranges, 0)
