"""GPU: every kernel behind the C-ABI, in isolation, against plain torch on the same device (fp32 math on the same
16-bit-rounded operands; fp16 unless the library was built with -DVITED_ACT_BF16=1). Tolerances are stated per test."""
import ctypes
import math

import pytest
import torch

pytestmark = pytest.mark.gpu


def _lib():
    from vited_b200 import _lib
    return _lib


def _act():
    return _lib().act_dtype()


def _r16():
    """tolerance scale of the 16-bit rounding terms: 1 for bf16 (8 significand bits), 0.2 for fp16 (11 bits)"""
    return 1.0 if _act() == torch.bfloat16 else 0.2


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _gemm(A, W, bias, act, impl):
    L = _lib()
    M, K = A.shape
    N = W.shape[0]
    C = torch.full((M, N), float('nan'), dtype=_act(), device='cuda')
    L.check(L.lib.vited_op_gemm(_ptr(A), _ptr(W), _ptr(bias), _ptr(C), M, N, K, act, impl, _stream()), 'op_gemm')
    torch.cuda.synchronize()
    return C


GEMM_SHAPES = [
    # (M, N, K): every Linear of the two models + ragged / tiny edge cases
    (128, 128, 64), (256, 384, 384), (1000, 1152, 384), (4160, 384, 384), (777, 1536, 384), (640, 384, 1536),
    (65 * 37, 768, 384), (64 * 9, 384, 192), (300, 384, 768), (5, 32, 32), (130, 96, 3072), (1, 8, 8),
    (129, 1152, 384), (20000, 1152, 384),
    # large M, K <= 384
    (30000, 1536, 384), (26000, 384, 384), (26001, 384, 192), (19999, 768, 384),
]


@pytest.mark.parametrize('impl', [0, 1], ids=['tcgen05', 'simt'])
@pytest.mark.parametrize('act', [0, 1], ids=['none', 'gelu'])
@pytest.mark.parametrize('shape', GEMM_SHAPES, ids=lambda s: 'x'.join(map(str, s)))
def test_gemm(shape, act, impl):
    M, N, K = shape
    if impl == 1 and M * N * K > 3e9:
        pytest.skip('debug kernel: skip the largest shape')
    g = torch.Generator(device='cuda').manual_seed(M * 7 + N * 3 + K)
    A = torch.randn(M, K, device='cuda', generator=g).to(_act())
    W = (torch.randn(N, K, device='cuda', generator=g) / math.sqrt(K)).to(_act())
    bias = torch.randn(N, device='cuda', generator=g)
    C = _gemm(A, W, bias, act, impl)
    ref = A.float() @ W.float().t() + bias
    if act:
        ref = torch.nn.functional.gelu(ref)
    assert torch.isfinite(C.float()).all(), 'output has NaN/inf (unwritten tile?)'
    # 16-bit output rounding (bf16 2^-9 / fp16 2^-12 relative) + fp32 accumulation-order noise
    err = (C.float() - ref).abs()
    tol = (1e-2 * ref.abs() + 2e-2) * _r16()
    bad = (err > tol)
    assert not bad.any(), f'{int(bad.sum())} / {bad.numel()} mismatches, max err {float(err.max()):.4f}, ' \
                          f'first bad index {bad.nonzero()[0].tolist()}'


def test_gelu_epilogue_accuracy():
    """The single-MUFU GELU of the GEMM epilogue against the exact erf definition (timm Mlp act_layer=nn.GELU) on a
    dense grid of pre-activations: |error| <= 1e-4 + the 16-bit rounding of the stored result."""
    M, N, K = 8192, 8, 8
    v = torch.linspace(-12, 12, M, device='cuda').to(_act())
    A = torch.zeros(M, K, dtype=_act(), device='cuda')
    A[:, 0] = v
    W = torch.eye(N, K, device='cuda').to(_act())
    bias = torch.zeros(N, device='cuda')
    C = _gemm(A, W, bias, 1, 0)
    ref = torch.nn.functional.gelu(v.double())
    err = (C[:, 0].double() - ref).abs()
    tol = 1e-4 + ref.abs() * (2.0 ** -8 if _act() == torch.bfloat16 else 2.0 ** -11)
    assert (err <= tol).all(), f'max excess {(err - tol).max().item()}'
    assert (C[:, 1:] == 0).all()


@pytest.mark.parametrize('bn', ['128', '192', '256'])
def test_gemm_tile_shapes_agree(bn):
    """Each tile width of the single-CTA tcgen05 kernel, picked by N (the widest of 256 / 192 / 128 that divides it),
    against torch."""
    M, N, K = {'128': (1111, 640, 384), '192': (1111, 1152, 384), '256': (1111, 1536, 384)}[bn]
    g = torch.Generator(device='cuda').manual_seed(1)
    A = torch.randn(M, K, device='cuda', generator=g).to(_act())
    W = (torch.randn(N, K, device='cuda', generator=g) / math.sqrt(K)).to(_act())
    b = torch.randn(N, device='cuda', generator=g)
    C = _gemm(A, W, b, 0, 0)
    ref = A.float() @ W.float().t() + b
    err = (C.float() - ref).abs().max().item()
    assert err < 0.06, err


def test_gemm_cta_pair_variant():
    """The cta_group::2 (CTA-pair) variant of the tcgen05 kernel, which takes M of at least two 128-row blocks per SM,
    against torch."""
    g = torch.Generator(device='cuda').manual_seed(1)
    for (M, N, K, act) in [(40000, 1536, 384, 1), (40001, 384, 1536, 0), (38001, 1152, 384, 0), (40000, 384, 384, 0),
                           (39990, 768, 384, 0)]:
        A = torch.randn(M, K, device='cuda', generator=g).to(_act())
        W = (torch.randn(N, K, device='cuda', generator=g) / math.sqrt(K)).to(_act())
        b = torch.randn(N, device='cuda', generator=g)
        C = _gemm(A, W, b, act, 0)
        ref = A.float() @ W.float().t() + b
        ref = torch.nn.functional.gelu(ref) if act else ref
        assert torch.isfinite(C.float()).all(), ('nan', M, N, K)
        err = (C.float() - ref).abs()
        tol = 1e-2 * ref.abs() + 2e-2
        bad = err > tol
        assert not bad.any(), (M, N, K, int(bad.sum()), float(err.max()), bad.nonzero()[0].tolist())


@pytest.mark.parametrize('D', [384, 768, 32, 96])
@pytest.mark.parametrize('has_cls', [0, 1])
def test_resid_ln(D, has_cls):
    L = _lib()
    n_seq, n_patch = 37, 9
    rows = n_seq * n_patch + (n_seq if has_cls else 0)
    g = torch.Generator(device='cuda').manual_seed(D + has_cls)
    x = torch.randn(rows, D, device='cuda', generator=g)
    delta = torch.randn(rows, D, device='cuda', generator=g).to(_act())
    w = 1 + 0.1 * torch.randn(D, device='cuda', generator=g)
    b = 0.1 * torch.randn(D, device='cuda', generator=g)
    x_ref = x + delta.float()
    h_ref = torch.nn.functional.layer_norm(x_ref, (D,), w, b, 1e-6)
    h = torch.zeros(rows, D, dtype=_act(), device='cuda')
    L.check(L.lib.vited_op_resid_ln(_ptr(x), _ptr(delta), _ptr(w), _ptr(b), _ptr(h), n_seq, n_patch, has_cls, D, 1e-6,
                                    _stream()), 'op_resid_ln')
    torch.cuda.synchronize()
    assert torch.equal(x, x_ref), 'residual update must be exact fp32'
    # 16-bit rounding of the normalised row
    assert (h.float() - h_ref).abs().max().item() <= (1e-2 * h_ref.abs().max().item() + 1e-3) * _r16()


@pytest.mark.parametrize('shape', [(256, 384), (70000, 384), (33333, 1536), (1, 384), (300, 64), (40000, 192)],
                         ids=lambda s: 'x'.join(map(str, s)))
def test_gemm_resid_ln_fused(shape):
    """x += A W^T + b; h = LayerNorm(x): the fused tcgen05 epilogue (8 warps x 192-column half rows) against fp32 torch
    on the same 16-bit operands."""
    L = _lib()
    M, K = shape
    N = 384
    g = torch.Generator(device='cuda').manual_seed(M + K)
    A = torch.randn(M, K, device='cuda', generator=g).to(_act())
    W = (torch.randn(N, K, device='cuda', generator=g) / math.sqrt(K)).to(_act())
    bias = torch.randn(N, device='cuda', generator=g)
    # rows with a large common offset exercise the shifted variance
    x = torch.randn(M, N, device='cuda', generator=g) * 2 + torch.randn(M, 1, device='cuda', generator=g) * 5
    lw = 1 + 0.1 * torch.randn(N, device='cuda', generator=g)
    lb = 0.1 * torch.randn(N, device='cuda', generator=g)
    x_ref = x + A.float() @ W.float().t() + bias
    h_ref = torch.nn.functional.layer_norm(x_ref, (N,), lw, lb, 1e-6)
    h = torch.full((M, N), float('nan'), dtype=_act(), device='cuda')
    L.check(L.lib.vited_op_gemm_resid_ln(_ptr(A), _ptr(W), _ptr(bias), _ptr(x), _ptr(lw), _ptr(lb), _ptr(h), M, N, K,
                                         1e-6, _stream()), 'op_gemm_resid_ln')
    torch.cuda.synchronize()
    assert torch.isfinite(h.float()).all() and torch.isfinite(x).all()
    # fp32 accumulation-order noise only (the accumulator is never rounded to 16 bits on this path)
    assert (x - x_ref).abs().max().item() < 1e-3 * max(1.0, x_ref.abs().max().item())
    # 16-bit rounding of the normalised row
    assert (h.float() - h_ref).abs().max().item() <= (1e-2 * h_ref.abs().max().item() + 2e-3) * _r16()


@pytest.mark.parametrize('shape', [(256, 1536), (70000, 1536), (33333, 1536), (1, 1536), (300, 64), (40000, 192),
                                   (262144 + 77, 1536)], ids=lambda s: 'x'.join(map(str, s)))
def test_mlp_resid_ln_fused(shape):
    """x += fc2(GELU(fc1(h))) + b2; h = LayerNorm(x): the fused MLP kernel (hidden activations kept in TMEM, GELU
    output fed to the second MMA as its A operand from TMEM) against fp32 torch on the same 16-bit operands, with the
    hidden activations rounded to 16 bits where the kernel rounds them. In place: h_out aliases h_in."""
    L = _lib()
    M, HID = shape
    D = 384
    g = torch.Generator(device='cuda').manual_seed(M + HID)
    h_in = torch.randn(M, D, device='cuda', generator=g).to(_act())
    W1 = (torch.randn(HID, D, device='cuda', generator=g) / math.sqrt(D)).to(_act())
    b1 = 0.5 * torch.randn(HID, device='cuda', generator=g)
    W2 = (torch.randn(D, HID, device='cuda', generator=g) / math.sqrt(HID)).to(_act())
    b2 = torch.randn(D, device='cuda', generator=g)
    x = torch.randn(M, D, device='cuda', generator=g) * 2 + torch.randn(M, 1, device='cuda', generator=g) * 5
    lw = 1 + 0.1 * torch.randn(D, device='cuda', generator=g)
    lb = 0.1 * torch.randn(D, device='cuda', generator=g)
    hid = torch.nn.functional.gelu(h_in.float() @ W1.float().t() + b1).to(_act()).float()
    x_ref = x + hid @ W2.float().t() + b2
    h_ref = torch.nn.functional.layer_norm(x_ref, (D,), lw, lb, 1e-6)
    h = h_in.clone()
    L.check(L.lib.vited_op_mlp_resid_ln(_ptr(h), _ptr(W1), _ptr(b1), _ptr(W2), _ptr(b2), _ptr(x), _ptr(lw), _ptr(lb),
                                        _ptr(h), M, D, HID, 1e-6, _stream()), 'op_mlp_resid_ln')
    torch.cuda.synchronize()
    assert torch.isfinite(h.float()).all() and torch.isfinite(x).all()
    # the hidden activations are rounded to 16 bits (as the unfused path stores them); a value next to a rounding
    # boundary may round the other way because of the GELU approximation (< 9e-5): a few 16-bit steps over K = hidden
    tol_x = (2e-3 if _act() == torch.float16 else 1.5e-2) * max(1.0, x_ref.abs().max().item())
    assert (x - x_ref).abs().max().item() < tol_x, (x - x_ref).abs().max().item()
    assert (h.float() - h_ref).abs().max().item() <= (1e-2 * h_ref.abs().max().item() + 4e-3) * _r16()


def _attn_reference(q, k, v, scale):
    # q [B,H,Nq,hd] etc, fp32 math on the 16-bit-rounded inputs
    s = (q.float() @ k.float().transpose(-1, -2)) * scale
    return s.softmax(dim=-1) @ v.float()


@pytest.mark.parametrize('impl', [0, 1, 2], ids=['fast', 'simt', 'mma_sync'])
@pytest.mark.parametrize('cfg', [
    # (n_seq, H, hd, n_patch, has_cls)  -- self-attention
    (7, 12, 32, 64, 1), (1, 1, 32, 64, 1), (333, 12, 32, 64, 1), (150, 5, 32, 64, 0), (3, 5, 32, 64, 1), (2000, 12, 32, 64, 1),
    (40, 6, 64, 1024, 1), (1, 1, 64, 256, 1), (9, 3, 64, 512, 0), (30, 2, 64, 256, 1), (3, 6, 64, 1024, 1), (5, 12, 32, 64, 0), (2, 6, 64, 1024, 0), (4, 1, 32, 4, 1),
    (3, 3, 32, 16, 1), (2, 2, 64, 100, 1), (1, 2, 32, 130, 0),
], ids=lambda c: 'x'.join(map(str, c)))
def test_self_attention(cfg, impl):
    L = _lib()
    n_seq, H, hd, n_patch, has_cls = cfg
    D = H * hd
    rows = n_seq * n_patch + (n_seq if has_cls else 0)
    g = torch.Generator(device='cuda').manual_seed(sum(cfg))
    qkv = torch.randn(rows, 3 * D, device='cuda', generator=g).to(_act())
    o = torch.full((rows, D), float('nan'), dtype=_act(), device='cuda')
    scale = hd ** -0.5
    st = L.lib.vited_op_attention(_ptr(qkv), 3 * D, ctypes.c_void_p(qkv.data_ptr() + 2 * D), 3 * D,
                                  ctypes.c_void_p(qkv.data_ptr() + 4 * D), 3 * D, _ptr(o), D, n_seq, H, hd, n_patch,
                                  has_cls, n_patch, has_cls, n_seq, None, scale, impl, _stream())
    L.check(st, 'op_attention')
    torch.cuda.synchronize()
    # reference in the logical [B, N, D] layout: token 0 = cls
    patch = qkv[:n_seq * n_patch].view(n_seq, n_patch, 3 * D)
    seq = torch.cat([qkv[n_seq * n_patch:].view(n_seq, 1, 3 * D), patch], dim=1) if has_cls else patch
    q, k, v = [seq[..., i * D:(i + 1) * D].reshape(n_seq, -1, H, hd).permute(0, 2, 1, 3) for i in range(3)]
    ref = _attn_reference(q, k, v, scale).permute(0, 2, 1, 3).reshape(n_seq, -1, D)
    got_patch = o[:n_seq * n_patch].view(n_seq, n_patch, D).float()
    got = torch.cat([o[n_seq * n_patch:].view(n_seq, 1, D).float(), got_patch], dim=1) if has_cls else got_patch
    assert torch.isfinite(got).all()
    # P is rounded to 16 bits before P.V and so is the output: 2e-2 (bf16) / 4e-3 (fp16) absolute on O(1) values
    assert (got - ref).abs().max().item() < 2e-2 * _r16(), f'max err {(got - ref).abs().max().item()}'


@pytest.mark.parametrize('impl', [0, 1, 2], ids=['fast', 'simt', 'mma_sync'])
@pytest.mark.parametrize('cfg', [
    # (n_pairs, n_ctx, H, hd, n_patch)
    (9, 4, 12, 32, 64), (1, 1, 12, 32, 64), (401, 7, 12, 32, 64), (7, 3, 5, 32, 64), (1500, 9, 12, 32, 64), (37, 5, 6, 64, 1024), (3, 2, 1, 64, 256), (5, 3, 6, 64, 1024), (6, 2, 1, 32, 4), (4, 4, 2, 64, 16),
], ids=lambda c: 'x'.join(map(str, c)))
def test_cross_attention(cfg, impl):
    L = _lib()
    P, n_ctx, H, hd, n_patch = cfg
    D = H * hd
    rows = P * (n_patch + 1)
    g = torch.Generator(device='cuda').manual_seed(sum(cfg))
    qb = torch.randn(rows, D, device='cuda', generator=g).to(_act())
    kv = torch.randn(n_ctx * n_patch, 2 * D, device='cuda', generator=g).to(_act())
    idx = torch.randint(0, n_ctx, (P,), device='cuda', generator=g, dtype=torch.int32)
    o = torch.full((rows, D), float('nan'), dtype=_act(), device='cuda')
    scale = hd ** -0.5
    st = L.lib.vited_op_attention(_ptr(qb), D, _ptr(kv), 2 * D, ctypes.c_void_p(kv.data_ptr() + 2 * D), 2 * D, _ptr(o),
                                  D, P, H, hd, n_patch, 1, n_patch, 0, n_ctx, _ptr(idx), scale, impl, _stream())
    L.check(st, 'op_attention')
    torch.cuda.synchronize()
    seq = torch.cat([qb[P * n_patch:].view(P, 1, D), qb[:P * n_patch].view(P, n_patch, D)], dim=1)
    q = seq.reshape(P, n_patch + 1, H, hd).permute(0, 2, 1, 3)
    kvs = kv.view(n_ctx, n_patch, 2, H, hd)[idx.long()]
    k = kvs[:, :, 0].permute(0, 2, 1, 3)
    v = kvs[:, :, 1].permute(0, 2, 1, 3)
    ref = _attn_reference(q, k, v, scale).permute(0, 2, 1, 3).reshape(P, n_patch + 1, D)
    got = torch.cat([o[P * n_patch:].view(P, 1, D), o[:P * n_patch].view(P, n_patch, D)], dim=1).float()
    assert torch.isfinite(got).all()
    assert (got - ref).abs().max().item() < 2e-2 * _r16(), f'max err {(got - ref).abs().max().item()}'


@pytest.mark.parametrize('impl', [0, 2], ids=['fast', 'mma_sync'])
def test_long_attention_lazy_rescale_paths(impl):
    """Scores that grow from key block to key block force the lazy rescale of the running maximum (and of the O row in
    TMEM) again and again; scores that shrink never trigger it. Both against fp32 torch. (Random-init weights and randn
    inputs never move a row maximum by more than the 2^8 threshold: until this test existed the rescale path had never
    run, and it hung -- warp-collective tcgen05 instructions under a per-thread condition.)"""
    L = _lib()
    n_seq, H, hd, n_patch = 3, 2, 64, 512
    D = H * hd
    rows = n_seq * n_patch + n_seq
    g = torch.Generator(device='cuda').manual_seed(5)
    for direction in (1.0, -1.0):
        qkv = torch.randn(rows, 3 * D, device='cuda', generator=g)
        # key magnitudes ramp over the sequence so that the row maxima move by far more than the 2^8 threshold
        ramp = torch.linspace(0.2, 6.0, n_patch, device='cuda')
        if direction < 0:
            ramp = ramp.flip(0)
        qkv[:n_seq * n_patch, D:2 * D] *= ramp.repeat(n_seq)[:, None]
        qkv[:, :D] *= 2.0
        qkv = qkv.to(_act())
        o = torch.full((rows, D), float('nan'), dtype=_act(), device='cuda')
        scale = hd ** -0.5
        L.check(L.lib.vited_op_attention(_ptr(qkv), 3 * D, ctypes.c_void_p(qkv.data_ptr() + 2 * D), 3 * D,
                                         ctypes.c_void_p(qkv.data_ptr() + 4 * D), 3 * D, _ptr(o), D, n_seq, H, hd, n_patch,
                                         1, n_patch, 1, n_seq, None, scale, impl, _stream()), 'op_attention')
        torch.cuda.synchronize()
        patch = qkv[:n_seq * n_patch].view(n_seq, n_patch, 3 * D)
        seq = torch.cat([qkv[n_seq * n_patch:].view(n_seq, 1, 3 * D), patch], dim=1)
        q, k, v = [seq[..., i * D:(i + 1) * D].reshape(n_seq, -1, H, hd).permute(0, 2, 1, 3) for i in range(3)]
        if direction > 0:   # the inputs must really move the row maxima by more than 2^8 between key blocks
            s_blocks = ((q.float() @ k.float().transpose(-1, -2)) * scale * 1.4426950408889634)[..., 1:].reshape(n_seq, H, -1, n_patch // 64, 64)
            assert (s_blocks.amax(-1)[..., -1] - s_blocks.amax(-1)[..., 0]).max().item() > 8.0
        ref = _attn_reference(q, k, v, scale).permute(0, 2, 1, 3).reshape(n_seq, -1, D)
        got = torch.cat([o[n_seq * n_patch:].view(n_seq, 1, D).float(), o[:n_seq * n_patch].view(n_seq, n_patch, D).float()], dim=1)
        assert torch.isfinite(got).all()
        assert (got - ref).abs().max().item() < 2e-2 * _r16(), f'max err {(got - ref).abs().max().item()}'


@pytest.mark.parametrize('cfg', [(3, 3, 64, 8), (2, 3, 512, 16), (5, 3, 64, 32)])
def test_im2col_patch_indexing_is_exact(cfg):
    L = _lib()
    B, C, S, p = cfg
    g = torch.Generator(device='cuda').manual_seed(0)
    img = torch.randn(B, C, S, S, device='cuda', generator=g)
    G = S // p
    out = torch.zeros(B * G * G, C * p * p, dtype=_act(), device='cuda')
    L.check(L.lib.vited_op_im2col(_ptr(img), _ptr(out), B, C, S, p, _stream()), 'op_im2col')
    torch.cuda.synchronize()
    ref = img.reshape(B, C, G, p, G, p).permute(0, 2, 4, 1, 3, 5).reshape(B * G * G, C * p * p).to(_act())
    assert torch.equal(out, ref), 'patch indexing must be bit-exact (SURVEY 8b)'


def test_fp16_results_saturate_instead_of_overflowing():
    """A 16-bit result beyond the fp16 range is stored as +-65504, not inf (the reference under autocast would carry
    inf / nan on); bf16 builds have the fp32 range and are not affected."""
    if _act() != torch.float16:
        pytest.skip('bf16 build')
    M, N, K = 512, 384, 64
    A = torch.full((M, K), 200.0, device='cuda').to(_act())
    W = torch.full((N, K), 200.0, device='cuda').to(_act())
    W[N // 2:] = -200.0
    C = _gemm(A, W, torch.zeros(N, device='cuda'), 0, 0)          # +-2.56e6 per element
    assert torch.isfinite(C.float()).all()
    assert (C[:, :N // 2].float() == 65504.0).all() and (C[:, N // 2:].float() == -65504.0).all()
    # fused Linear + residual + LayerNorm: the fp32 residual takes the full value, the normalised row stays finite
    L = _lib()
    x = torch.zeros(M, N, device='cuda')
    h = torch.full((M, N), float('nan'), dtype=_act(), device='cuda')
    lw, lb = torch.full((N,), 1e6, device='cuda'), torch.zeros(N, device='cuda')
    L.check(L.lib.vited_op_gemm_resid_ln(_ptr(A), _ptr(W), _ptr(torch.zeros(N, device='cuda')), _ptr(x), _ptr(lw),
                                         _ptr(lb), _ptr(h), M, N, K, 1e-6, _stream()), 'op_gemm_resid_ln')
    torch.cuda.synchronize()
    assert (x[:, 0] == 200.0 * 200.0 * K).all()
    assert torch.isfinite(h.float()).all() and (h.float().abs() == 65504.0).all()
