"""GPU: scoring caller-given pair lists (vited_score_pairs(_u8), model.score_pairs, grid.score_pairs) and extending a
scored fragment collection (grid.extend_fragments). A dense grid's own pair set in its i-major order must give the
grid's bits; any other list must give the grid's entries up to the fp32 noise of other chunk shapes and stay on the
fp32 oracle; only the items a list references may be computed."""
import ctypes
import os

import numpy as np
import pytest
import torch

from tests import helpers
from tests.test_gpu_fragment_scale import _restore, _to_u8

pytestmark = pytest.mark.gpu

TIGHT = 4e-3          # tests/test_gpu_parity.py: fp16 operands against the fp32 oracle
SENTINEL = 12345.0


@pytest.fixture(scope='module')
def puzzle_case():
    from oracle import vited_oracle as orc
    from vited_b200 import synthetic
    z, kw = helpers.load_model_case('puzzle_patch8_64')
    model, sd = helpers.make_gpu_model(kw, 3)
    images = synthetic.synthetic_images(37, kw['img_size'], seed=31)
    want12 = orc.score_puzzle_grid(sd, kw['num_heads'], images[:12])       # fp32, CPU: ordered pairs of items < 12
    return model, kw, images.cuda(), _to_u8(images), want12


@pytest.fixture(scope='module')
def hisfrag_case():
    from oracle import vited_oracle as orc
    from vited_b200 import synthetic
    z, kw = helpers.load_model_case('hisfrag20_patch16_512')
    model, sd = helpers.make_gpu_model(kw, 5)
    images, labels = synthetic.synthetic_fragments(4, 2, kw['img_size'], seed=3)
    want = orc.score_fragment_grid(sd, kw['num_heads'], images)          # fp32, CPU: score(a, b) at [a, b] and [b, a]
    return model, kw, images.cuda(), _to_u8(images), want


def _grid_pairs(mode, n, lo, hi):
    """the grid's pair set of rows [lo, hi), i-major with j ascending"""
    import vited_b200
    from vited_b200 import grid
    full = grid.ordered_pairs(n) if mode == vited_b200.GRID_ORDERED_OFFDIAG else grid.upper_tri_pairs(n)
    return full[(full[:, 0] >= lo) & (full[:, 0] < hi)]


def _random_pairs(n, count, seed):
    """shuffled, with duplicates, a == b and a > b"""
    rng = np.random.default_rng(seed)
    p = rng.integers(0, n, size=(count, 2)).astype(np.int32)
    p[:5, 1] = p[:5, 0]                               # a == b
    p = np.concatenate([p, p[:7], p[10:13, ::-1]])    # duplicates, reversed pairs
    return p[rng.permutation(len(p))]


def _dense_reference(model, images, pairs):
    """the (a, b) entry of the ordered grid, or the upper-triangular grid's diagonal when a == b"""
    import vited_b200
    ordered = model.score_grid(images, vited_b200.GRID_ORDERED_OFFDIAG)
    upper = model.score_grid(images, vited_b200.GRID_UPPER_TRI_DIAG)
    a = torch.from_numpy(pairs[:, 0]).long().cuda()
    b = torch.from_numpy(pairs[:, 1]).long().cuda()
    return torch.where((a == b)[:, None], upper[a, b], ordered[a, b])


# ------------------------------------------------------------------------------------------------------------ dense
@pytest.mark.parametrize('case,mode_name,rows', [
    ('puzzle', 'ordered', None), ('puzzle', 'ordered', (5, 19)), ('puzzle', 'upper', None), ('puzzle', 'upper', (5, 19)),
    ('hisfrag', 'upper', None), ('hisfrag', 'upper', (2, 7)), ('hisfrag', 'ordered', None)])
def test_dense_grid_as_a_pair_list_is_bit_identical(puzzle_case, hisfrag_case, case, mode_name, rows):
    import vited_b200
    model, kw, f32, u8 = (puzzle_case if case == 'puzzle' else hisfrag_case)[:4]
    mode = vited_b200.GRID_ORDERED_OFFDIAG if mode_name == 'ordered' else vited_b200.GRID_UPPER_TRI_DIAG
    _restore(model)
    n = u8.shape[0]
    lo, hi = rows if rows else (0, n)
    pairs = _grid_pairs(mode, n, lo, hi)
    dense = model.score_grid(u8, mode, lo, hi)
    got = model.score_pairs(u8, torch.from_numpy(pairs).cuda())
    want = dense[torch.from_numpy(pairs[:, 0] - lo).long().cuda(), torch.from_numpy(pairs[:, 1]).long().cuda()]
    assert torch.equal(got, want)


# ------------------------------------------------------------------------------------------------------------ lists
def test_arbitrary_list_puzzle_model(puzzle_case):
    model, kw, f32, u8, want12 = puzzle_case
    _restore(model)
    pairs = _random_pairs(37, 300, 1)
    small = _random_pairs(12, 60, 2)                  # items the oracle covers
    pairs = np.concatenate([pairs, small])
    got = model.score_pairs(u8, torch.from_numpy(pairs).cuda())
    assert got.shape == (len(pairs), 4)
    assert (got - _dense_reference(model, u8, pairs)).abs().max().item() < 2e-3
    tail = got[-len(small):].cpu()
    off = small[:, 0] != small[:, 1]
    err = (tail[off] - want12[small[off, 0], small[off, 1]]).abs().max().item()
    assert err < TIGHT, err


def test_arbitrary_list_hisfrag_model(hisfrag_case):
    model, kw, f32, u8, want = hisfrag_case
    _restore(model)
    pairs = _random_pairs(8, 40, 3)
    got = model.score_pairs(f32, torch.from_numpy(pairs).long().cuda())      # int64 pairs
    assert (got - _dense_reference(model, f32, pairs)).abs().max().item() < 2e-3
    up = pairs[:, 0] <= pairs[:, 1]                   # the oracle matrix holds score(a, b) for a <= b
    err = (got[:, 0].cpu()[up] - want[pairs[up, 0], pairs[up, 1]]).abs().max().item()
    assert err < TIGHT, err


@pytest.mark.parametrize('case,kv_mb,xsrc_mb', [('puzzle', 1, 1), ('hisfrag', 40, 2)])
def test_forced_budgets_split_the_list_into_cells(puzzle_case, hisfrag_case, case, kv_mb, xsrc_mb):
    """puzzle: 1 MB of K/V = one context item per block, 1 MB of decoder states = 10 items per window;
    Hisfrag: 40 MB of K/V = two fragments per block, 2 MB = one fragment per window."""
    import vited_b200
    model, kw, f32, u8 = (puzzle_case if case == 'puzzle' else hisfrag_case)[:4]
    n = u8.shape[0]
    pairs = torch.from_numpy(_random_pairs(n, 150 if case == 'puzzle' else 40, 4)).cuda()
    _restore(model)
    one = model.score_pairs(u8, pairs)
    model.set_option(vited_b200.OPT_KV_BUDGET_MB, kv_mb)
    model.set_option(vited_b200.OPT_XSRC_BUDGET_MB, xsrc_mb)
    cells = model.score_pairs(u8, pairs)
    _restore(model)
    assert (cells - one).abs().max().item() < 2e-3
    p = pairs.cpu().numpy()
    if case == 'hisfrag':
        want = hisfrag_case[4]
        up = p[:, 0] <= p[:, 1]
        err = (cells[:, 0].cpu()[up] - want[p[up, 0], p[up, 1]]).abs().max().item()
    else:
        want12 = puzzle_case[4]
        sel = (p[:, 0] < 12) & (p[:, 1] < 12) & (p[:, 0] != p[:, 1])
        err = (cells.cpu()[sel] - want12[p[sel, 0], p[sel, 1]]).abs().max().item()
    assert err < TIGHT, err


def test_uint8_equals_fp32_on_the_same_list(puzzle_case, hisfrag_case):
    for model, kw, f32, u8 in (puzzle_case[:4], hisfrag_case[:4]):
        _restore(model)
        pairs = torch.from_numpy(_random_pairs(u8.shape[0], 80, 5)).cuda()
        assert torch.equal(model.score_pairs(u8, pairs), model.score_pairs(f32, pairs))


@pytest.mark.parametrize('fmt', ['u8', 'f32'])
def test_only_referenced_items_are_computed(puzzle_case, fmt):
    """3 context items and 5 decoder items out of 37: the patch matrices formed cover exactly those 8 items."""
    import vited_b200
    model, kw, f32, u8, _ = puzzle_case
    _restore(model)
    images = u8 if fmt == 'u8' else f32
    ctx, dec = [4, 17, 30], [0, 4, 9, 22, 36]
    pairs = torch.tensor([[a, b] for a in ctx for b in dec] + [[17, 22]], dtype=torch.int32, device='cuda')
    model.set_option(vited_b200.OPT_PROFILE, 1)
    try:
        model.score_pairs(images, pairs)
        prof = model.profile_read()
    finally:
        model.set_option(vited_b200.OPT_PROFILE, 0)
    n_e, k_pe = (kw['img_size'] // kw['patch_size']) ** 2, 3 * kw['patch_size'] ** 2
    per_item = n_e * k_pe * (3.0 if fmt == 'u8' else 6.0)
    name = 'im2col_u8' if fmt == 'u8' else 'im2col'
    assert prof[name]['bytes'] == pytest.approx((len(ctx) + len(dec)) * per_item, rel=1e-9)
    assert 'pair_index' in prof


# ------------------------------------------------------------------------------------------------------------ errors
@pytest.mark.parametrize('bad', [37, -1, 2 ** 40])
def test_out_of_range_index_is_an_error_before_scoring(puzzle_case, bad):
    import vited_b200
    model, kw, f32, u8, _ = puzzle_case
    _restore(model)
    pairs = torch.tensor([[0, 1], [2, 3], [4, 5], [6, bad], [bad, 1], [7, 8]], dtype=torch.int64, device='cuda')
    out = torch.full((6, 4), SENTINEL, dtype=torch.float32, device='cuda')
    with pytest.raises(vited_b200.VitedError) as err:
        model.score_pairs(u8, pairs, out=out)
    assert 'pair 3 ' in str(err.value) and '(2 such pairs)' in str(err.value), str(err.value)
    torch.cuda.synchronize()
    assert (out == SENTINEL).all()
    assert torch.equal(model.score_pairs(u8, pairs[:3]), model.score_pairs(u8, pairs[:3]))   # the engine still works


def test_empty_list_is_a_no_op(puzzle_case):
    from vited_b200 import _lib
    model, kw, f32, u8, _ = puzzle_case
    out = model.score_pairs(u8, torch.zeros((0, 2), dtype=torch.int32, device='cuda'))
    assert out.shape == (0, 4)
    sentinel = torch.full((1, 4), SENTINEL, device='cuda')
    rc = _lib.lib.vited_score_pairs_u8(model._ensure_engine(u8.device), u8.data_ptr(), u8.shape[0], None, 0,
                                       sentinel.data_ptr(), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == 0 and (sentinel == SENTINEL).all()


def test_bad_pair_tensors_raise_value_error(puzzle_case):
    model, kw, f32, u8, _ = puzzle_case
    with pytest.raises(ValueError):
        model.score_pairs(u8, torch.zeros((3, 2), dtype=torch.int32))                          # on the CPU
    with pytest.raises(ValueError):
        model.score_pairs(u8, torch.zeros((3, 3), dtype=torch.int32, device='cuda'))           # wrong shape
    with pytest.raises(ValueError):
        model.score_pairs(u8, torch.zeros(6, dtype=torch.int32, device='cuda'))
    with pytest.raises(ValueError):
        model.score_pairs(u8, torch.zeros((3, 2), dtype=torch.float32, device='cuda'))         # wrong dtype


# ------------------------------------------------------------------------------------------------------------ extension
def test_extend_fragments_matches_the_full_rescore(hisfrag_case):
    from vited_b200 import grid
    model, kw, f32, u8, want = hisfrag_case
    _restore(model)
    is_new = np.zeros(8, dtype=bool)
    is_new[[1, 4, 6]] = True
    old = np.flatnonzero(~is_new)
    full = grid.score_fragments(model, f32)
    for images in (f32, u8):
        old_sim = grid.score_fragments(model, images[torch.from_numpy(old).cuda()])
        ext = grid.extend_fragments(model, images, old_sim, is_new)
        assert ext.shape == (8, 8)
        o = torch.from_numpy(old).cuda()
        assert torch.equal(ext[o[:, None], o[None, :]], old_sim)
        assert (ext - full).abs().max().item() < 2e-3
        assert (ext.cpu() - want).abs().max().item() < TIGHT
    with pytest.raises(ValueError):
        grid.extend_fragments(model, f32, old_sim[:4, :4], is_new)


def test_retrieval_metrics_after_extension():
    """The mixed retrieval fixture: 40 fragments scored, then extended by the other 8 (at interleaved positions),
    gives the metrics of the full re-score to 3 decimals."""
    import vited_b200
    from tests.test_gpu_retrieval import _retrieval_case
    from vited_b200 import grid
    z, kw, sd, images, labels, sim_orc, m_stored = _retrieval_case('mixed')
    model = vited_b200.VisionTransformerCustom(mlp_ratio=4., qkv_bias=True, **kw)
    model.load_state_dict(sd, strict=True)
    model = model.cuda().eval()
    images = images.cuda()
    n = images.shape[0]
    is_new = np.zeros(n, dtype=bool)
    is_new[np.random.default_rng(8).choice(n, 8, replace=False)] = True
    old_sim = grid.score_fragments(model, images[torch.from_numpy(np.flatnonzero(~is_new)).cuda()])
    ext = grid.extend_fragments(model, images, old_sim, is_new)
    base = grid.retrieval_metrics(grid.score_fragments(model, images), labels)
    got = grid.retrieval_metrics(ext, labels)
    for a, b in zip(got, base):
        assert round(a, 3) == round(b, 3), (got, base)


# ------------------------------------------------------------------------------------------------------------ 2 ranks
def _worker(rank, world, port, q):
    import torch.distributed as dist
    import vited_b200
    from vited_b200 import grid, synthetic
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group('nccl', rank=rank, world_size=world, device_id=torch.device('cuda', rank))
    try:
        z, kw = helpers.load_model_case('small_hd64')
        model, _ = helpers.make_gpu_model(kw, 2)
        images = synthetic.synthetic_images(23, kw['img_size'], seed=9).cuda()
        pairs = _random_pairs(23, 200, 6)
        scores = grid.score_pairs(model, images, pairs)
        is_new = np.zeros(23, dtype=bool)
        is_new[[0, 7, 8, 22]] = True
        old = images[torch.from_numpy(np.flatnonzero(~is_new)).cuda()]
        old_sim = grid.mirror_upper(model.score_grid(old, vited_b200.GRID_UPPER_TRI_DIAG)[..., 0])   # no collective
        ext = grid.extend_fragments(model, images, old_sim, is_new)
        q.put((rank, scores.cpu(), ext.cpu()))
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs two GPUs')
def test_two_rank_pair_lists_and_extension_equal_single_gpu():
    import torch.multiprocessing as mp
    from vited_b200 import grid, synthetic
    world = 2
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = 29600 + (os.getpid() + 11) % 2000
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    results = [q.get(timeout=600) for _ in range(world)]
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    z, kw = helpers.load_model_case('small_hd64')
    model, _ = helpers.make_gpu_model(kw, 2)
    images = synthetic.synthetic_images(23, kw['img_size'], seed=9).cuda()
    single = model.score_pairs(images, torch.from_numpy(_random_pairs(23, 200, 6)).cuda()).cpu()
    full = grid.score_fragments(model, images).cpu()
    for rank, scores, ext in results:
        assert (scores - single).abs().max().item() < 1e-2, rank
        assert (ext - full).abs().max().item() < 1e-2, rank
