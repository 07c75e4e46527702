"""CPU: grid.hisfrag_row_ranges, the closed form of the Hisfrag row sharding, against the pair-list computation it
replaces (grid.indicates_row_ranges over upper_tri_pairs, the reference's DistributedIndicatesSampler) and against the
sampler vectors the reference produced."""
import os
import time

import numpy as np
import pytest

from tests.conftest import GOLDEN


def _reference(n, world):
    from vited_b200 import grid
    return grid.indicates_row_ranges(grid.upper_tri_pairs(n)[:, 0], world)


def test_closed_form_equals_pair_list_form_small_grids():
    from vited_b200 import grid
    for n in range(1, 401):
        for world in range(1, 17):
            assert grid.hisfrag_row_ranges(n, world) == _reference(n, world), (n, world)


@pytest.mark.parametrize('world', [2, 3, 5, 7, 8])
def test_closed_form_equals_pair_list_form_up_to_3000(world):
    from vited_b200 import grid
    for n in list(range(401, 3001, 37)) + [1000, 2047, 2048, 2049, 3000]:
        assert grid.hisfrag_row_ranges(n, world) == _reference(n, world), (n, world)


def test_closed_form_matches_reference_sampler_vectors():
    from vited_b200 import grid
    z = np.load(os.path.join(GOLDEN, 'integer_paths.npz'))
    for n, world in z['sampler_cases']:
        n, world = int(n), int(world)
        sizes = grid.hisfrag_row_ranges(n, world)
        assert sizes == _reference(n, world)
        ref = z[f'sampler_{n}_{world}']
        for rank in range(world):
            if ref[rank, 0] == -2:
                assert rank + 1 >= len(sizes)
            else:
                assert [sizes[rank], sizes[rank + 1]] == ref[rank].tolist()


def test_empty_grid_fails_like_the_reference():
    from vited_b200 import grid
    with pytest.raises(ValueError):
        _reference(0, 2)
    with pytest.raises(ValueError):
        grid.hisfrag_row_ranges(0, 2)


def test_large_grid_is_fast_and_covers_every_row():
    from vited_b200 import grid
    t0 = time.perf_counter()
    sizes = grid.hisfrag_row_ranges(50_000, 8)
    assert time.perf_counter() - t0 < 0.1
    assert sizes[0] == 0 and sizes[-1] == 50_000 and len(sizes) == 9
    assert all(a < b for a, b in zip(sizes, sizes[1:]))
    # every rank's share of the 1.25 G pairs is the equal split to within two rows
    n = 50_000
    per = [(hi - lo) * n - (hi * (hi - 1) - lo * (lo - 1)) // 2 for lo, hi in zip(sizes, sizes[1:])]
    assert sum(per) == n * (n + 1) // 2
    assert max(per) - min(per) <= 2 * n, per
