"""CPU: the host side of pair-list scoring -- the extension pairs of a grown fragment collection and the sharding of a
pair list over ranks with its reassembly in input order."""
import numpy as np
import pytest
import torch


def _masks():
    rng = np.random.default_rng(11)
    yield np.zeros(7, dtype=bool)                     # no new items
    yield np.ones(9, dtype=bool)                      # all items new
    first = np.zeros(12, dtype=bool)
    first[0] = True
    yield first
    last = np.zeros(12, dtype=bool)
    last[-1] = True
    yield last
    yield np.array([True], dtype=bool)
    for n in (2, 5, 31, 64, 200):
        for p in (0.05, 0.3, 0.8):
            yield rng.random(n) < p


@pytest.mark.parametrize('is_new', list(_masks()), ids=lambda m: f'n{len(m)}_new{int(m.sum())}')
def test_extension_pairs_is_the_upper_triangle_minus_old_pairs(is_new):
    from vited_b200 import grid
    n = len(is_new)
    got = grid.extension_pairs(is_new)
    assert got.dtype == np.int32 and got.shape[1] == 2
    full = grid.upper_tri_pairs(n)
    keep = is_new[full[:, 0]] | is_new[full[:, 1]]
    np.testing.assert_array_equal(got, full[keep])     # same set, same a-major / b-ascending order
    n_new = int(is_new.sum())
    assert len(got) == (n - n_new) * n_new + n_new * (n_new + 1) // 2


@pytest.mark.parametrize('world', range(1, 9))
@pytest.mark.parametrize('n_pairs', [0, 1, 3, 7, 50, 1001])
def test_pair_shares_round_trip(world, n_pairs):
    from vited_b200 import grid
    rng = np.random.default_rng(world * 1000 + n_pairs)
    ctx = rng.integers(0, 13, size=n_pairs)
    order, bounds = grid.pair_shares(ctx, world)
    assert len(bounds) == world + 1 and bounds[0] == 0 and bounds[-1] == n_pairs
    assert all(a <= b for a, b in zip(bounds, bounds[1:]))
    sizes = np.diff(bounds)
    assert sizes.max(initial=0) - sizes.min(initial=0) <= max(1, -(-n_pairs // world))
    assert sorted(order.tolist()) == list(range(n_pairs))
    sorted_ctx = ctx[order]
    assert (np.diff(sorted_ctx) >= 0).all()
    for c in np.unique(ctx):                          # stable: input order kept among equal context items
        pos = order[sorted_ctx == c]
        assert (np.diff(pos) > 0).all()
    # every rank "scores" its share: value = input position, padded to the longest share with garbage
    longest = max(int(sizes.max(initial=0)), 1)
    gathered = torch.full((world, longest, 2), -7.0)
    for r in range(world):
        share = order[bounds[r]:bounds[r + 1]]
        gathered[r, :len(share), 0] = torch.from_numpy(share).float()
        gathered[r, :len(share), 1] = torch.from_numpy(ctx[share]).float()
    out = grid.unpermute_shares(gathered, order, bounds)
    assert out.shape == (n_pairs, 2)
    np.testing.assert_array_equal(out[:, 0].numpy(), np.arange(n_pairs))
    np.testing.assert_array_equal(out[:, 1].numpy(), ctx)


def test_pair_shares_with_fewer_pairs_than_ranks_leave_ranks_empty():
    from vited_b200 import grid
    order, bounds = grid.pair_shares(np.array([4, 1, 4]), 5)
    assert bounds == [0, 1, 2, 3, 3, 3]
    assert order.tolist() == [1, 0, 2]
