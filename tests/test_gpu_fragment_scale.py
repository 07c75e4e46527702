"""GPU: the fragment grid at dataset scale -- uint8 crops straight into the patch matrix (vited_op_im2col_u8,
vited_score_grid_u8) and the decoder input states of the grid columns held in bounded windows
(OPT_XSRC_BUDGET_MB). The uint8 path must be bit-identical to the fp32 path on the images the bytes normalise to;
the windowed grid must equal the one-window grid up to the fp32 noise of other chunk shapes and stay on the oracle."""
import ctypes
import os

import numpy as np
import pytest
import torch

from tests import helpers

pytestmark = pytest.mark.gpu

TIGHT = 4e-3          # tests/test_gpu_parity.py: fp16 operands against the fp32 oracle
SENTINEL = 12345.0


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _normalize(u8):
    """[N, S, S, 3] uint8 (CUDA) -> [N, 3, S, S] fp32 through vited_normalize_u8"""
    from vited_b200 import _lib
    n, s = u8.shape[0], u8.shape[1]
    out = torch.empty((n, 3, s, s), dtype=torch.float32, device='cuda')
    _lib.check(_lib.lib.vited_normalize_u8(_ptr(u8), n, s, _ptr(out), _stream()), 'vited_normalize_u8')
    return out


def _to_u8(images):
    """fp32 [N, 3, S, S] in [-1, 1] built from bytes (synthetic.*) -> those bytes as CUDA [N, S, S, 3]; asserts that
    the bytes normalise back to exactly the given floats, so the two forms are the same input."""
    u8 = torch.round((images.float() * 0.5 + 0.5) * 255.0).clamp(0, 255).to(torch.uint8)
    u8 = u8.permute(0, 2, 3, 1).contiguous().cuda()
    assert torch.equal(_normalize(u8).cpu(), images.cpu()), 'the synthetic images are not exact byte images'
    return u8


def _restore(model):
    import vited_b200
    for opt, val in ((vited_b200.OPT_KV_BUDGET_MB, 8000), (vited_b200.OPT_XSRC_BUDGET_MB, 32000)):
        model.set_option(opt, val)


# ------------------------------------------------------------------------------------------------------------ kernel
@pytest.mark.parametrize('S,p', [(64, 8), (512, 16)])
def test_im2col_u8_is_bit_identical_to_normalize_then_im2col(S, p):
    from vited_b200 import _lib
    B, C = 3, 3
    g = torch.Generator().manual_seed(S + p)
    u8 = torch.randint(0, 256, (B, S, S, C), generator=g, dtype=torch.uint8)
    u8.view(-1)[:256 * 3] = torch.arange(256, dtype=torch.uint8).repeat_interleave(3)   # every byte in every channel
    u8 = u8.cuda()
    K, rows = C * p * p, B * (S // p) ** 2
    want = torch.full((rows, K), float('nan'), dtype=_lib.act_dtype(), device='cuda')
    got = torch.full((rows, K), float('nan'), dtype=_lib.act_dtype(), device='cuda')
    f32 = _normalize(u8)
    _lib.check(_lib.lib.vited_op_im2col(_ptr(f32), _ptr(want), B, C, S, p, _stream()), 'vited_op_im2col')
    _lib.check(_lib.lib.vited_op_im2col_u8(_ptr(u8), _ptr(got), B, C, S, p, _stream()), 'vited_op_im2col_u8')
    assert torch.equal(got, want)
    assert len(torch.unique(got)) == 256


def test_im2col_u8_rejects_shapes_it_has_no_kernel_for():
    from vited_b200 import _lib
    u8 = torch.zeros((1, 48, 48, 3), dtype=torch.uint8, device='cuda')
    out = torch.empty((9, 3 * 16 * 16), dtype=_lib.act_dtype(), device='cuda')
    assert _lib.lib.vited_op_im2col_u8(_ptr(u8), _ptr(out), 1, 3, 48, 12, _stream()) != 0
    assert 'no kernel' in _lib.last_error()


# ------------------------------------------------------------------------------------------------------------ grids
@pytest.fixture(scope='module')
def puzzle_case():
    from vited_b200 import synthetic
    z, kw = helpers.load_model_case('puzzle_patch8_64')
    model, sd = helpers.make_gpu_model(kw, 3)
    images = synthetic.synthetic_images(37, kw['img_size'], seed=31)
    return model, kw, images.cuda(), _to_u8(images)


@pytest.fixture(scope='module')
def hisfrag_case():
    from oracle import vited_oracle as orc
    from vited_b200 import synthetic
    z, kw = helpers.load_model_case('hisfrag20_patch16_512')
    model, sd = helpers.make_gpu_model(kw, 5)
    images, labels = synthetic.synthetic_fragments(4, 2, kw['img_size'], seed=3)
    want = orc.score_fragment_grid(sd, kw['num_heads'], images)          # fp32, CPU
    return model, kw, images.cuda(), _to_u8(images), want


def test_uint8_grid_equals_fp32_grid_puzzle_model(puzzle_case):
    import vited_b200
    model, kw, f32, u8 = puzzle_case
    _restore(model)
    mode = vited_b200.GRID_ORDERED_OFFDIAG
    assert torch.equal(model.score_grid(u8, mode), model.score_grid(f32, mode))
    assert torch.equal(model.score_grid(u8, mode, 5, 19), model.score_grid(f32, mode, 5, 19))


def test_uint8_grid_equals_fp32_grid_hisfrag_model(hisfrag_case):
    import vited_b200
    from vited_b200 import grid
    model, kw, f32, u8, want = hisfrag_case
    _restore(model)
    mode = vited_b200.GRID_UPPER_TRI_DIAG
    full = model.score_grid(u8, mode)
    assert torch.equal(full, model.score_grid(f32, mode))
    assert torch.equal(model.score_grid(u8, mode, 2, 7), model.score_grid(f32, mode, 2, 7))
    sim = grid.score_fragments(model, u8)
    assert torch.equal(sim, grid.score_fragments(model, f32))
    assert (sim.cpu() - want).abs().max().item() < TIGHT


def test_score_fragments_on_uploaded_crops_equals_the_fp32_batch(hisfrag_case):
    """pieces.fragments_to_u8_device (crop on the host, one upload of the bytes) feeds score_fragments, also through
    the resumable path, with the scores of fragments_to_batch_device's fp32 batch."""
    from vited_b200 import grid, pieces
    model, kw, _, _, _ = hisfrag_case
    _restore(model)
    rng = np.random.default_rng(4)
    raw = [rng.integers(0, 256, size=s + (3,), dtype=np.uint8) for s in [(600, 530), (512, 512), (515, 700), (400, 900)]]
    u8 = pieces.fragments_to_u8_device(raw, kw['img_size'])
    f32 = pieces.fragments_to_batch_device(raw, kw['img_size'])
    assert u8.dtype == torch.uint8 and u8.shape == (4, 512, 512, 3) and u8.is_cuda
    assert torch.equal(_normalize(u8), f32)
    want = grid.score_fragments(model, f32)
    assert torch.equal(grid.score_fragments(model, u8), want)


def test_score_fragments_resumable_path_takes_uint8(hisfrag_case, tmp_path):
    from vited_b200 import grid
    model, kw, f32, u8, _ = hisfrag_case
    _restore(model)
    want = grid.score_fragments(model, f32)
    got = grid.score_fragments(model, u8, resume_path=str(tmp_path / 'r{rank}.pt'), block_rows=3, save_every=1)
    np.testing.assert_allclose(got.cpu().numpy(), want.cpu().numpy(), rtol=0, atol=2e-3)


def test_score_grid_rejects_other_uint8_layouts(puzzle_case):
    import vited_b200
    model, kw, f32, u8 = puzzle_case
    with pytest.raises(ValueError):
        model.score_grid(u8.permute(0, 3, 1, 2), vited_b200.GRID_ORDERED_OFFDIAG)       # [N, C, S, S] bytes
    with pytest.raises(ValueError):
        model.score_grid(u8.cpu(), vited_b200.GRID_ORDERED_OFFDIAG)


# ------------------------------------------------------------------------------------------------------------ windows
def _sentinel_grid(model, images, mode, lo, hi):
    n = images.shape[0]
    out = torch.full((hi - lo, n, model.num_classes), SENTINEL, dtype=torch.float32, device='cuda')
    return model.score_grid(images, mode, lo, hi, out=out)


def _pair_mask(mode, n, lo, hi):
    import vited_b200
    i = torch.arange(lo, hi)[:, None]
    j = torch.arange(n)[None, :]
    return (j != i) if mode == vited_b200.GRID_ORDERED_OFFDIAG else (j >= i)


@pytest.mark.parametrize('mode_name', ['ordered', 'upper'])
@pytest.mark.parametrize('kv_mb,rows', [(None, None), (1, None), (1, (5, 30))])
def test_column_windows_puzzle_model(puzzle_case, mode_name, kv_mb, rows):
    """1 MB of column states = 10 puzzle items per window (65 tokens x 384 x 4 bytes each)."""
    import vited_b200
    model, kw, f32, u8 = puzzle_case
    mode = vited_b200.GRID_ORDERED_OFFDIAG if mode_name == 'ordered' else vited_b200.GRID_UPPER_TRI_DIAG
    n = u8.shape[0]
    lo, hi = rows if rows else (0, n)
    _restore(model)
    if kv_mb:
        model.set_option(vited_b200.OPT_KV_BUDGET_MB, kv_mb)
    one = _sentinel_grid(model, u8, mode, lo, hi)
    model.set_option(vited_b200.OPT_XSRC_BUDGET_MB, 1)
    windows = _sentinel_grid(model, u8, mode, lo, hi)
    _restore(model)
    mask = _pair_mask(mode, n, lo, hi).cuda()
    assert (windows[~mask] == SENTINEL).all() and (one[~mask] == SENTINEL).all()
    assert (windows[mask] != SENTINEL).all()
    err = (windows[mask] - one[mask]).abs().max().item()
    assert err < 2e-3, err


@pytest.mark.parametrize('kv_mb,rows', [(None, (0, 8)), (40, (0, 8)), (40, (2, 7))])
def test_column_windows_hisfrag_model(hisfrag_case, kv_mb, rows):
    """2 MB of column states = one Hisfrag fragment (1,025 tokens x 384 x 4 bytes) per window; with 40 MB of K/V
    budget the rows come in blocks of two fragments."""
    import vited_b200
    model, kw, f32, u8, want = hisfrag_case
    mode = vited_b200.GRID_UPPER_TRI_DIAG
    n = u8.shape[0]
    lo, hi = rows
    _restore(model)
    if kv_mb:
        model.set_option(vited_b200.OPT_KV_BUDGET_MB, kv_mb)
    one = _sentinel_grid(model, u8, mode, lo, hi)
    model.set_option(vited_b200.OPT_XSRC_BUDGET_MB, 2)
    windows = _sentinel_grid(model, u8, mode, lo, hi)
    _restore(model)
    mask = _pair_mask(mode, n, lo, hi).cuda()
    assert (windows[~mask] == SENTINEL).all()
    assert (windows[mask] - one[mask]).abs().max().item() < 2e-3
    err = (windows[..., 0].cpu() - want[lo:hi])[mask.cpu()].abs().max().item()
    assert err < TIGHT, err


def test_budget_covering_all_columns_keeps_the_launch_sequence(hisfrag_case):
    """A budget at or above the call's column states is the one-window path: the same scores bit for bit and the
    same number of launches as the default."""
    import vited_b200
    model, kw, f32, u8, want = hisfrag_case
    mode = vited_b200.GRID_UPPER_TRI_DIAG
    n = u8.shape[0]
    _restore(model)
    n0 = model.launch_count()
    default = model.score_grid(u8, mode)
    d_default = model.launch_count() - n0
    per_item = 1025 * 384 * 4
    model.set_option(vited_b200.OPT_XSRC_BUDGET_MB, -(-n * per_item // 1_000_000))      # just enough for all columns
    n0 = model.launch_count()
    exact = model.score_grid(u8, mode)
    d_exact = model.launch_count() - n0
    model.set_option(vited_b200.OPT_XSRC_BUDGET_MB, 2)
    n0 = model.launch_count()
    model.score_grid(u8, mode)
    d_windows = model.launch_count() - n0
    _restore(model)
    assert torch.equal(exact, default) and d_exact == d_default
    assert d_windows > d_default          # the states really were rebuilt per window


def test_retrieval_metrics_through_uint8_and_column_windows():
    """The mixed retrieval fixture (tests/test_gpu_retrieval.py) scored from bytes with 1 MB of column states (two
    fragments per window) gives the metrics of the fp32 one-window path to 3 decimals."""
    import vited_b200
    from tests.test_gpu_retrieval import _retrieval_case
    from vited_b200 import grid
    z, kw, sd, images, labels, sim_orc, m_stored = _retrieval_case('mixed')
    model = vited_b200.VisionTransformerCustom(mlp_ratio=4., qkv_bias=True, **kw)
    model.load_state_dict(sd, strict=True)
    model = model.cuda().eval()
    base = grid.retrieval_metrics(grid.score_fragments(model, images.cuda()), labels)
    sim = grid.score_fragments(model, _to_u8(images), xsrc_budget_mb=1)
    got = grid.retrieval_metrics(sim, labels)
    for a, b in zip(got, base):
        assert round(a, 3) == round(b, 3), (got, base)


# ------------------------------------------------------------------------------------------------------------ 2 ranks
def _worker(rank, world, port, q):
    import torch.distributed as dist
    from vited_b200 import grid, synthetic
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group('nccl', rank=rank, world_size=world, device_id=torch.device('cuda', rank))
    try:
        z, kw = helpers.load_model_case('small_hd64')
        model, _ = helpers.make_gpu_model(kw, 2)
        images = synthetic.synthetic_images(23, kw['img_size'], seed=9)
        u8 = torch.round((images * 0.5 + 0.5) * 255.0).to(torch.uint8).permute(0, 2, 3, 1).contiguous().cuda()
        sim = grid.score_fragments(model, u8, xsrc_budget_mb=1)
        q.put((rank, sim.cpu()))
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs two GPUs')
def test_two_rank_uint8_fragments_with_column_windows_equal_single_gpu():
    import torch.multiprocessing as mp
    from vited_b200 import grid, synthetic
    world = 2
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = 29600 + (os.getpid() + 7) % 2000
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
    single = grid.score_fragments(model, images).cpu()
    for rank, sim in results:
        assert (sim - single).abs().max().item() < 1e-2, rank
