"""GPU: the 13 training-step entry points (``vited_train_*``, csrc/train_ops.cu and csrc/train_attn.cu) one by one
against a float64 torch computation of the same operation on the same 16-bit-rounded inputs, at the Hisfrag20 sizes
(1,024 encoder / 1,025 decoder tokens, 24 images, 72 pairs) and at the edges where kernels go wrong: ragged tails,
single rows, grid-stride loops, remainder loops.

Every test that writes a buffer also checks what it must leave alone: accumulating outputs start from a random
non-zero prefill and the test compares ``result - prefill``; rows past the logical end of every output hold a NaN
sentinel that must survive.

Tolerances are written in units of u, the unit roundoff of the 16-bit type the library was built with (2^-11 for
fp16, 2^-8 for -DVITED_ACT_BF16=1 builds), and of 2^-24 for fp32 arithmetic. Each test's docstring derives its bound
from the roundings the kernel does and quotes the largest error measured on a B200 (fp16 build, bf16 build)."""
import ctypes
import math
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu

GUARD = 3           # NaN sentinel rows after the logical end of every output buffer
E32 = 2.0 ** -24    # fp32 unit roundoff


def _lib():
    from vited_b200 import _lib
    return _lib


def _act():
    return _lib().act_dtype()


def _u16():
    """unit roundoff of the 16-bit activation type: 2^-8 (bf16, 8 significand bits) or 2^-11 (fp16, 11 bits)"""
    return 2.0 ** -8 if _act() == torch.bfloat16 else 2.0 ** -11


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _gen(seed):
    return torch.Generator(device='cuda').manual_seed(seed)


def _guarded(t):
    """(buffer, view): ``t`` followed by GUARD rows of NaN in one buffer; the view is the first t.shape[0] rows"""
    buf = torch.full((t.shape[0] + GUARD,) + tuple(t.shape[1:]), float('nan'), dtype=t.dtype, device=t.device)
    buf[:t.shape[0]] = t
    return buf, buf[:t.shape[0]]


def _assert_guard(buf, n, what):
    assert torch.isnan(buf[n:].float()).all(), f'{what}: the rows past the end of the output were written'


def _to16(x):
    """x.to(act) with the kernels' f2act rule: fp16 saturates at +-65504 instead of overflowing to inf"""
    if _act() == torch.float16:
        x = x.clamp(-65504.0, 65504.0)
    return x.to(_act())


def _report(name, **errs):
    print(f'[{_act()}] {name}: ' + ', '.join(f'{k} {v:.3g}' for k, v in errs.items()))


def _status_fails(status, what):
    assert status != 0, f'{what}: expected a non-zero status'
    msg = _lib().last_error()
    assert msg, f'{what}: failed without a message'
    return msg


# ---------------------------------------------------------------------------------------------------------------
# 1. attention (train_attn.cu: wmma, head_dim 32 / 64; train_ops.cu: SIMT reference, any head_dim multiple of 8)
# ---------------------------------------------------------------------------------------------------------------
# (name, n_seq, H, hd, Tq, Tk, layout): 'self' = q / k / v column slices of one [rows, 3D] buffer (ld 3D), 'cross' = q
# its own [rows, D] buffer, k / v column slices of a [rows, 2D] buffer -- as train.py lays them out
ATTN_CASES = [
    ('hisfrag_encoder_self', 2, 6, 64, 1024, 1024, 'self'),
    ('hisfrag_decoder_self', 2, 6, 64, 1025, 1025, 'self'),
    ('hisfrag_cross', 3, 6, 64, 1025, 1024, 'cross'),
    ('hd32_blocks', 3, 12, 32, 65, 64, 'cross'),
    ('hd32_ragged', 2, 2, 32, 63, 129, 'cross'),
    ('single_token', 1, 1, 64, 1, 1, 'self'),
    ('tk_gt_tq', 1, 3, 64, 64, 65, 'cross'),
    ('tq_gt_tk', 1, 1, 32, 200, 7, 'cross'),
    ('simt_auto_hd16', 2, 4, 16, 100, 100, 'self'),
    ('simt_auto_hd48', 2, 3, 48, 70, 130, 'cross'),
]
SIMT_FORCED = ['hisfrag_decoder_self', 'hisfrag_cross', 'hd32_blocks', 'hd32_ragged']


def _simt_selected(hd):
    return os.environ.get('VITED_TRAIN_ATTN_SIMT', '0') not in ('', '0') or hd not in (32, 64)


def _attn_inputs(n_seq, H, hd, Tq, Tk, layout, seed, q_gain=1.0, ramp=0):
    """16-bit q / k / v views in train.py's layout, fp32 d_o. ``ramp`` = +1 / -1 scales the keys by a magnitude that
    grows / shrinks over the sequence, so the row maximum of the scores moves from key block to key block."""
    D = H * hd
    g = _gen(seed)
    if layout == 'self':
        assert Tq == Tk
        base = torch.randn(n_seq * Tq, 3 * D, device='cuda', generator=g)
        q32, k32 = base[:, :D], base[:, D:2 * D]
    else:
        qbase = torch.randn(n_seq * Tq, D, device='cuda', generator=g)
        base = torch.randn(n_seq * Tk, 2 * D, device='cuda', generator=g)
        q32, k32 = qbase, base[:, :D]
    q32.mul_(q_gain)
    if ramp:
        r = torch.linspace(0.2, 6.0, Tk, device='cuda')
        k32.mul_((r if ramp > 0 else r.flip(0)).repeat(n_seq)[:, None])
    if layout == 'self':
        b16 = base.to(_act())
        q, k, v = b16[:, :D], b16[:, D:2 * D], b16[:, 2 * D:]
    else:
        q = qbase.to(_act())
        b16 = base.to(_act())
        k, v = b16[:, :D], b16[:, D:]
    d_o = torch.randn(n_seq * Tq, D, device='cuda', generator=g)
    return dict(shape=(n_seq, H, hd, Tq, Tk), layout=layout, q=q, k=k, v=v, d_o=d_o, scale=hd ** -0.5, seed=seed)


def _attn_call(c, backward, o, lse, d_o=None, dsum=None, dq=None, dk=None, dv=None):
    L = _lib()
    n_seq, H, hd, Tq, Tk = c['shape']
    ld = lambda t: t.stride(0) if t is not None else 0
    return L.lib.vited_train_attention(int(backward), _ptr(c['q']), ld(c['q']), _ptr(c['k']), ld(c['k']), _ptr(c['v']),
                                       ld(c['v']), _ptr(o), ld(o), _ptr(lse), _ptr(d_o), ld(d_o), _ptr(dsum), _ptr(dq),
                                       ld(dq), _ptr(dk), ld(dk), _ptr(dv), ld(dv), n_seq, H, hd, Tq, Tk, c['scale'],
                                       _stream())


def _attn_run(c, pass_o_to_backward=True):
    """Forward, then backward from the forward's o and lse; returns the outputs (gradients as result - prefill, in
    float64) after checking every NaN sentinel."""
    L = _lib()
    n_seq, H, hd, Tq, Tk = c['shape']
    D = H * hd
    rq, rk, nl = n_seq * Tq, n_seq * Tk, n_seq * H * Tq
    g = _gen(c['seed'] + 1)
    nan = float('nan')
    o_buf = torch.full((rq + GUARD, D), nan, dtype=_act(), device='cuda')
    lse_buf = torch.full((nl + GUARD,), nan, device='cuda')
    o, lse = o_buf[:rq], lse_buf[:nl]
    L.check(_attn_call(c, 0, o, lse), 'train_attention forward')
    dsum_buf = torch.full((nl + GUARD,), nan, device='cuda')
    if c['layout'] == 'self':
        gbuf, _ = _guarded(torch.randn(rq, 3 * D, device='cuda', generator=g))
        dq, dk, dv = gbuf[:rq, :D], gbuf[:rq, D:2 * D], gbuf[:rq, 2 * D:]
        bufs = [(gbuf, rq, 'dqkv')]
    else:
        qbuf, _ = _guarded(torch.randn(rq, D, device='cuda', generator=g))
        kvbuf, _ = _guarded(torch.randn(rk, 2 * D, device='cuda', generator=g))
        dq, dk, dv = qbuf[:rq], kvbuf[:rk, :D], kvbuf[:rk, D:]
        bufs = [(qbuf, rq, 'dq'), (kvbuf, rk, 'dkv')]
    pre = [t.double() for t in (dq, dk, dv)]
    L.check(_attn_call(c, 1, o if pass_o_to_backward else None, lse, c['d_o'], dsum_buf[:nl], dq, dk, dv),
            'train_attention backward')
    torch.cuda.synchronize()
    _assert_guard(o_buf, rq, 'o')
    _assert_guard(lse_buf, nl, 'lse')
    _assert_guard(dsum_buf, nl, 'dsum')
    for buf, n, what in bufs:
        _assert_guard(buf, n, what)
    return dict(o=o.double(), lse=lse.double(), dsum=dsum_buf[:nl].double(), dq=dq.double() - pre[0],
                dk=dk.double() - pre[1], dv=dv.double() - pre[2])


def _attn_reference(c):
    """float64 autograd of softmax(q k^T * scale) v on the kernel's 16-bit inputs, in the kernel's row layouts"""
    n_seq, H, hd, Tq, Tk = c['shape']

    def heads(t, T):
        return t.double().reshape(n_seq, T, H, hd).transpose(1, 2).contiguous().requires_grad_()

    q, k, v = heads(c['q'], Tq), heads(c['k'], Tk), heads(c['v'], Tk)
    do = c['d_o'].double().reshape(n_seq, Tq, H, hd).transpose(1, 2)
    with torch.enable_grad():
        s = (q @ k.transpose(-1, -2)) * c['scale']
        o = torch.softmax(s, dim=-1) @ v
        o.backward(do)
    rows = lambda t, T: t.detach().transpose(1, 2).reshape(n_seq * T, H * hd)
    return dict(o=rows(o, Tq), lse=torch.logsumexp(s.detach(), dim=-1).reshape(-1),
                dsum=(do * o.detach()).sum(-1).reshape(-1), dq=rows(q.grad, Tq), dk=rows(k.grad, Tk),
                dv=rows(v.grad, Tk), s=s.detach())


def _attn_tolerances(c, simt):
    """Bounds of the attention outputs; see test_attention_matches_float64_autograd for the derivation."""
    n_seq, H, hd, Tq, Tk = c['shape']
    u = _u16()
    qn = c['q'].double().reshape(-1, hd).norm(dim=-1).max().item()
    kn = c['k'].double().reshape(-1, hd).norm(dim=-1).max().item()
    e_s = hd * 2.0 ** -23 * c['scale'] * qn * kn               # fp32 (tensor-core) accumulation error of a score
    vmax = c['v'].double().abs().max().item()
    e_sum = (Tk + 64) * 2.0 ** -23                             # fp32 sums over the keys
    if simt:
        return dict(o=(u + 2 * e_s + e_sum) * vmax, lse=e_s + e_sum, grad=SIMT_GRAD_TOL)
    return dict(o=(3 * u + 2 * e_s + e_sum) * vmax, lse=u + e_s + e_sum, grad=WMMA_GRAD_TOL * u)


WMMA_GRAD_TOL = 8      # dq / dk / dv of the wmma kernels, relative to the max of each tensor, in units of u
SIMT_GRAD_TOL = 2e-5   # the same for the fp32 SIMT kernels (no 16-bit rounding inside)


def _attn_errors(c, got, ref, simt):
    tol = _attn_tolerances(c, simt)
    n_seq, H, hd, Tq, Tk = c['shape']
    do_abs = c['d_o'].double().abs().reshape(n_seq, Tq, H, hd).transpose(1, 2).sum(-1).reshape(-1)
    if Tk == 1:
        # one key: the softmax is constant, dq = dk = 0 exactly, and the kernels return the rounding noise of
        # dS = p (dP - D) scale (dO and o rounded to 16 bits, fp32 dot products), times |k| or |q|
        qk = max(c['q'].double().abs().max().item(), c['k'].double().abs().max().item())
        noise = c['scale'] * (3 * _u16() + hd * 2.0 ** -23) * do_abs.max().item() * \
            c['v'].double().abs().max().item() * qk
        floor = noise / tol['grad']
    else:
        floor = 1e-30
    rel = lambda k: ((got[k] - ref[k]).abs().max() / ref[k].abs().max().clamp_min(floor)).item()
    lse_err = (got['lse'] - ref['lse']).abs() - 2.0 ** -22 * ref['lse'].abs()
    # D_i = do_i . o_i: the o error above, weighted by sum |do_i|
    dsum_excess = ((got['dsum'] - ref['dsum']).abs() - do_abs * tol['o']).max().item()
    errs = dict(o=(got['o'] - ref['o']).abs().max().item(), lse=lse_err.max().item(), dsum_excess=dsum_excess,
                dq=rel('dq'), dk=rel('dk'), dv=rel('dv'))
    return errs, tol


def _attn_assert(name, c, got, ref, simt):
    errs, tol = _attn_errors(c, got, ref, simt)
    _report(f'attention {name} ({"simt" if simt else "wmma"})', o=errs['o'], o_tol=tol['o'], lse=errs['lse'],
            lse_tol=tol['lse'], dq=errs['dq'], dk=errs['dk'], dv=errs['dv'], grad_tol=tol['grad'])
    for key in ('o', 'dq', 'dk', 'dv', 'lse', 'dsum'):
        assert torch.isfinite(got[key]).all(), f'{name}: {key} has NaN / inf'
    assert errs['o'] <= tol['o'], f'{name}: o off by {errs["o"]:.3g} > {tol["o"]:.3g}'
    assert errs['lse'] <= tol['lse'], f'{name}: lse off by {errs["lse"]:.3g} > {tol["lse"]:.3g}'
    assert errs['dsum_excess'] <= 0, f'{name}: dsum exceeds its bound by {errs["dsum_excess"]:.3g}'
    for key in ('dq', 'dk', 'dv'):
        assert errs[key] <= tol['grad'], f'{name}: {key} off by {errs[key]:.3g} of its max > {tol["grad"]:.3g}'


@pytest.mark.parametrize('case', ATTN_CASES, ids=[c[0] for c in ATTN_CASES])
def test_attention_matches_float64_autograd(case):
    """Forward (o, lse) and backward (dsum, dq, dk, dv accumulated onto a random prefill) against float64 autograd of
    softmax(q k^T * scale) v on the same 16-bit q / k / v and fp32 d_o.

    Bounds. A score carries at most e_s = hd * 2^-23 * scale * |q| |k| of fp32 (tensor-core) accumulation error.
    wmma forward: P is rounded to 16 bits before P V, and the row sum is taken over the rounded P, so o moves by at most
    2u max|v|; the stored o adds u |o| <= u max|v|: |o - ref| <= (3u + 2 e_s + (Tk + 64) 2^-23) max|v|. lse comes from
    the sum of the rounded P (relative error <= u, fp16 subnormal P included in the Tk term): |lse - ref| <= u + e_s +
    (Tk + 64) 2^-23 + 2^-22 |lse|. SIMT: only o is rounded (u max|v|), P stays fp32. dsum = do . o: the o bound
    weighted by sum |do|. Backward: the wmma kernels round P, dS and dO to 16 bits before their MMAs and take D from
    the 16-bit o, so every product term carries about 3u: max error <= 8u of each tensor's max (fp16 and bf16); the
    SIMT kernels are fp32 throughout: <= 2e-5 of the max.
    Measured on a B200, largest over the cases (fp16 / bf16 build): wmma o 8.2e-4 / 5.2e-3 (bound >= 4.2e-3 /
    3.2e-2), lse 1.8e-4 / 1.1e-3, dq / dk / dv 5.2e-4 / 4.2e-3 of the max (1.1u / 1.1u); SIMT o 4.8e-4 / 3.7e-3 (the
    rounding of o), dq / dk / dv 2.0e-6 / 1.3e-6 of the max."""
    name, n_seq, H, hd, Tq, Tk, layout = case
    c = _attn_inputs(n_seq, H, hd, Tq, Tk, layout, seed=sum(case[1:6]))
    got = _attn_run(c)
    ref = _attn_reference(c)
    _attn_assert(name, c, got, ref, _simt_selected(hd))


@pytest.mark.parametrize('hd', [32, 64])
@pytest.mark.parametrize('direction', [1, -1], ids=['maxima_grow', 'maxima_shrink'])
def test_attention_online_softmax_rescale(direction, hd):
    """Key magnitudes ramp over the sequence (as in test_long_attention_lazy_rescale_paths), so the running row
    maximum of the wmma forward moves by e^8 and more between the first and the last full one of the 17 key blocks:
    growing maxima take the alpha = exp(m_run - m_new) rescale at every block, shrinking ones never do. Same bounds as
    test_attention_matches_float64_autograd (the score error e_s grows with |k|). Measured on a B200 (shrinking
    maxima): o 1.9e-3, dq / dk / dv 1.3e-3 of the max (fp16); o 1.5e-2, gradients 9.9e-3 (bf16)."""
    n_seq, H, T = 2, 3, 1025
    c = _attn_inputs(n_seq, H, hd, T, T, 'self', seed=40 + hd + direction, q_gain=2.0, ramp=direction)
    got = _attn_run(c)
    ref = _attn_reference(c)
    nb = (T + 63) // 64
    s = ref['s']
    bmax = torch.stack([s[..., j * 64:(j + 1) * 64].amax(-1) for j in range(nb)], dim=-1)   # [n_seq, H, T, blocks]
    move = (bmax[..., T // 64 - 1] - bmax[..., 0]) * direction          # last full block against the first
    assert move.median().item() > 8.0, f'the inputs do not move the row maxima enough ({move.median().item():.2f})'
    _attn_assert(f'rescale dir {direction} hd {hd}', c, got, ref, _simt_selected(hd))


def test_attention_sharp_softmax():
    """q scaled by 4: a typical row puts a third of its weight on one key of 1,025 (a flat row 1/1025). There the
    wmma backward's D = do . o, formed from the 16-bit o, differs most from sum_j p_j dP_j, and dP - D cancels for the
    dominant key. Same bounds. Measured on a B200: o 1.1e-3, dq / dk / dv 8.1e-4 of the max (fp16); o 8.7e-3,
    gradients 6.7e-3 (bf16)."""
    c = _attn_inputs(2, 6, 64, 1025, 1025, 'self', seed=77, q_gain=4.0)
    got = _attn_run(c)
    ref = _attn_reference(c)
    pmax = torch.softmax(ref['s'], dim=-1).amax(-1)
    assert pmax.median().item() > 0.25, 'the softmax is not sharp'
    _attn_assert('sharp', c, got, ref, _simt_selected(64))


def test_attention_wmma_backward_needs_o():
    """The tensor-core backward takes D = do . o from the forward's o: without it the call fails with a message and
    writes nothing."""
    if _simt_selected(64):
        pytest.skip('SIMT attention selected for this process')
    c = _attn_inputs(1, 2, 64, 65, 65, 'self', seed=3)
    n = 2 * 65
    lse = torch.zeros(n, device='cuda')
    dsum = torch.full((n,), float('nan'), device='cuda')
    dqkv = torch.full((65, 3 * 128), float('nan'), device='cuda')
    st = _attn_call(c, 1, None, lse, c['d_o'], dsum, dqkv[:, :128], dqkv[:, 128:256], dqkv[:, 256:])
    msg = _status_fails(st, 'wmma backward without o')
    assert 'needs o' in msg, msg
    torch.cuda.synchronize()
    assert torch.isnan(dqkv).all() and torch.isnan(dsum).all()


def _simt_child(out_dir):
    """Runs in a subprocess with VITED_TRAIN_ATTN_SIMT=1 (read once per process): the SIMT kernels at head_dim 32 / 64
    against float64 autograd; saves their outputs for the comparison with the wmma kernels."""
    assert _simt_selected(64)
    for case in ATTN_CASES:
        if case[0] not in SIMT_FORCED:
            continue
        name, n_seq, H, hd, Tq, Tk, layout = case
        c = _attn_inputs(n_seq, H, hd, Tq, Tk, layout, seed=sum(case[1:6]))
        got = _attn_run(c, pass_o_to_backward=False)      # the SIMT backward does not read o
        _attn_assert(name, c, got, _attn_reference(c), True)
        torch.save({k: v.cpu() for k, v in got.items()}, os.path.join(out_dir, f'{name}.pt'))


def test_simt_attention_at_hd32_and_hd64(tmp_path):
    """The SIMT reference kernels (train_ops.cu), forced with VITED_TRAIN_ATTN_SIMT=1 in a subprocess, against
    float64 autograd (fp32 bounds), and against the wmma kernels of this process on the same inputs: o within the wmma
    bound, gradients within the wmma bound of each tensor's max. Measured on a B200: SIMT against wmma o 9.8e-4,
    gradients 5.0e-4 of the max (fp16); o 3.9e-3, gradients 4.2e-3 (bf16)."""
    if _simt_selected(64):
        pytest.skip('SIMT attention selected for this process: no wmma results to compare with')
    from tests.conftest import ROOT
    code = f'import sys; sys.path.insert(0, {ROOT!r}); from tests import test_gpu_train_kernels as t; ' \
           f't._simt_child({str(tmp_path)!r})'
    env = dict(os.environ, VITED_TRAIN_ATTN_SIMT='1')
    r = subprocess.run([sys.executable, '-c', code], env=env, capture_output=True, text=True, timeout=600)
    print(r.stdout)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    for case in ATTN_CASES:
        if case[0] not in SIMT_FORCED:
            continue
        name, n_seq, H, hd, Tq, Tk, layout = case
        c = _attn_inputs(n_seq, H, hd, Tq, Tk, layout, seed=sum(case[1:6]))
        simt = {k: v.cuda() for k, v in torch.load(tmp_path / f'{name}.pt').items()}
        wmma = _attn_run(c)
        tol = _attn_tolerances(c, False)
        o_diff = (simt['o'] - wmma['o']).abs().max().item()
        rel = {k: ((simt[k] - wmma[k]).abs().max() / simt[k].abs().max()).item() for k in ('dq', 'dk', 'dv')}
        _report(f'attention {name} simt vs wmma', o=o_diff, **rel)
        assert o_diff <= tol['o'], f'{name}: SIMT and wmma o differ by {o_diff:.3g}'
        for k, e in rel.items():
            assert e <= tol['grad'], f'{name}: SIMT and wmma {k} differ by {e:.3g} of the max'


# ---------------------------------------------------------------------------------------------------------------
# 2. LayerNorm
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('D', [384, 128, 32, 100])
@pytest.mark.parametrize('R', [1, 31, 24576, 73800])
def test_layernorm_forward_backward(R, D):
    """train_ln_forward (stats, h) and train_ln_backward (dx, dw, db accumulated, alpha != 1) against float64
    layer_norm and its autograd, eps 1e-6. Every third row has a large common offset (mean 50, std 1). 73,800 rows
    (72 pairs x 1,025 tokens) need more blocks than the backward's 296-block grid, so each block folds many rows into
    its shared-memory partial sums.

    Bounds, with k = ceil(D / 32) + 8 (a lane's strided sum plus the 5-level warp reduction and a few roundings):
    mean <= k 2^-24 mean|x|; rstd relative <= k 2^-24; the normalised value xhat = (x - mean) rstd then carries
    e_xh = k 2^-24 (1 + |xhat| + |mean| rstd); h <= u |h| + |w| e_xh + 2^-24 (|b| + 1). dx = rstd (g - mean g - xhat
    mean(g xhat)), g = dh w: <= (k + 2) 2^-24 rstd (|g| + mean|g| + (|xhat| + e_xh) mean|g xhat|) + rstd mean|g| e_xh
    + 2^-24 |dx|. dw, db: sums over R rows, R / grid rows per block in shared memory then one atomic per block onto
    the prefill: <= (R / grid + grid + 4) 2^-24 (|prefill| + |alpha| sum |term|) + |alpha| sum |dh| e_xh.
    Measured on a B200, as a fraction of these bounds (fp16 and bf16 alike except h): mean 0.24, rstd 0.30, h 0.997
    (the 16-bit rounding itself), dx 0.35, dw 0.064, db 0.25; dx is within 1.6e-6 of its max."""
    L = _lib()
    g = _gen(R * 7 + D)
    u = _u16()
    x = torch.randn(R, D, device='cuda', generator=g) * 2.0
    x[::3] = 50.0 + torch.randn(x[::3].shape, device='cuda', generator=g)
    w = 1.0 + 0.1 * torch.randn(D, device='cuda', generator=g)
    b = 0.1 * torch.randn(D, device='cuda', generator=g)
    nan = float('nan')
    h_buf = torch.full((R + GUARD, D), nan, dtype=_act(), device='cuda')
    st_buf = torch.full((R + GUARD, 2), nan, device='cuda')
    L.check(L.lib.vited_train_ln_forward(_ptr(x), _ptr(w), _ptr(b), _ptr(h_buf), _ptr(st_buf), R, D, 1e-6, _stream()),
            'train_ln_forward')
    dh = torch.randn(R, D, device='cuda', generator=g)
    dx_buf, dx = _guarded(torch.randn(R, D, device='cuda', generator=g))
    dw_buf, dw = _guarded(torch.randn(D, device='cuda', generator=g))
    db_buf, db = _guarded(torch.randn(D, device='cuda', generator=g))
    pre = [t.double() for t in (dx, dw, db)]
    alpha = 0.37
    L.check(L.lib.vited_train_ln_backward(_ptr(dh), _ptr(x), _ptr(st_buf), _ptr(w), _ptr(dx), _ptr(dw), _ptr(db), R, D,
                                          alpha, _stream()), 'train_ln_backward')
    torch.cuda.synchronize()
    for buf, what in ((h_buf, 'h'), (st_buf, 'stats'), (dx_buf, 'dx')):
        _assert_guard(buf, R, what)
    for buf, what in ((dw_buf, 'dw'), (db_buf, 'db')):
        _assert_guard(buf, D, what)

    xl, w64, b64, dh64 = x.double().requires_grad_(), w.double().requires_grad_(), b.double().requires_grad_(), dh.double()
    with torch.enable_grad():
        h_ref = torch.nn.functional.layer_norm(xl, (D,), w64, b64, 1e-6)
        h_ref.backward(dh64)
    x64 = xl.detach()
    mean = x64.mean(-1, keepdim=True)
    rstd = (x64.var(-1, unbiased=False, keepdim=True) + 1e-6).rsqrt()
    xh = (x64 - mean) * rstd
    k = math.ceil(D / 32) + 8
    e_xh = k * E32 * (1 + xh.abs() + mean.abs() * rstd)
    stats = st_buf[:R].double()
    err_mean = ((stats[:, 0:1] - mean).abs() / (k * E32 * x64.abs().mean(-1, keepdim=True))).max().item()
    err_rstd = ((stats[:, 1:2] / rstd - 1).abs() / (k * E32)).max().item()
    h = h_buf[:R].double()
    tol_h = u * h_ref.detach().abs() + w64.detach().abs() * e_xh + E32 * (b64.detach().abs() + 1)
    err_h = ((h - h_ref.detach()).abs() / tol_h).max().item()

    gg = dh64 * w64.detach()
    mg = gg.abs().mean(-1, keepdim=True)
    mgx = (gg * xh).abs().mean(-1, keepdim=True)
    tol_dx = (k + 2) * E32 * rstd * (gg.abs() + mg + (xh.abs() + e_xh) * mgx) + rstd * mg * e_xh \
        + E32 * dx.double().abs()
    err_dx = ((dx.double() - pre[0] - xl.grad).abs() / tol_dx).max().item()
    grid = min(max((R * 32 + 255) // 256, 1), 296)
    depth = (R + grid - 1) // grid + grid + 4
    sum_dh = dh64.abs().sum(0)
    tol_dw = depth * E32 * (pre[1].abs() + alpha * (dh64 * xh).abs().sum(0)) + alpha * (dh64.abs() * e_xh).sum(0)
    tol_db = depth * E32 * (pre[2].abs() + alpha * sum_dh)
    err_dw = ((dw.double() - pre[1] - alpha * w64.grad).abs() / tol_dw).max().item()
    err_db = ((db.double() - pre[2] - alpha * b64.grad).abs() / tol_db).max().item()
    rel = lambda a, r: ((a - r).abs().max() / r.abs().max()).item()
    _report(f'layernorm R {R} D {D} (errors / bound)', mean=err_mean, rstd=err_rstd, h=err_h, dx=err_dx, dw=err_dw,
            db=err_db, h_rel=rel(h, h_ref.detach()), dx_rel=rel(dx.double() - pre[0], xl.grad))
    for key, e in (('mean', err_mean), ('rstd', err_rstd), ('h', err_h), ('dx', err_dx), ('dw', err_dw), ('db', err_db)):
        assert e <= 1.0, f'R {R} D {D}: {key} exceeds its bound {e:.3g}x'


# ---------------------------------------------------------------------------------------------------------------
# 3. GELU
# ---------------------------------------------------------------------------------------------------------------
def _all_16bit_values_in(lo, hi):
    bits = torch.arange(-32768, 32768, dtype=torch.int32, device='cuda').to(torch.int16)
    v = bits.view(_act())
    v = v[torch.isfinite(v.float()) & (v.float() >= lo) & (v.float() <= hi)]
    return v


@pytest.mark.parametrize('n', [1, 257, 2_000_003])
def test_gelu_forward_backward(n):
    """train_gelu_forward (16-bit z -> 16-bit a) against the exact erf GELU, and train_gelu_backward (dz = da *
    (Phi(z) + z phi(z))) in float64, on every 16-bit value in [-12, 12] plus random values; 2,000,003 elements are more
    than the 148 x 16 x 256-thread grid, so the grid-stride loop runs.

    Bounds: the fp32 gelu_erf = 0.5 z (1 + erff(z / sqrt 2)) is within 2^-24 (2|z| + |a|) of the exact value (erff
    <= 2 ulp, 1 + erf rounded), then the result is rounded to 16 bits: |a - gelu| <= u |gelu| + 2^-24 (2|z| + |a|) +
    2^-25 (fp16 subnormals). Backward, all fp32: Phi is within 2^-22 absolute, z phi(z) within 5 ulp, the sum and the
    product round once each: |dz - ref| <= |da| 2^-24 (4 + 5 |z phi| + 2 |gelu'|) + 2^-24 |dz|. Measured on a B200,
    as a fraction of the bounds: forward 1.0 (fp16) / 0.975 (bf16) -- the 16-bit rounding itself, |error| <= 9.8e-4 /
    7.8e-3 -- and backward 0.40 / 0.38."""
    L = _lib()
    g = _gen(n)
    grid = _all_16bit_values_in(-12.0, 12.0)
    rnd = (torch.randn(n, device='cuda', generator=g) * 4.0).to(_act())
    if n <= grid.numel():   # small n: a random half of the grid, then random values
        grid = grid[torch.randperm(grid.numel(), device='cuda', generator=g)[:n // 2]]
    z = torch.cat([grid, rnd])[:n].contiguous()
    assert z.numel() == n
    a_buf = torch.full((n + GUARD,), float('nan'), dtype=_act(), device='cuda')
    L.check(L.lib.vited_train_gelu_forward(_ptr(z), _ptr(a_buf), n, _stream()), 'train_gelu_forward')
    da = torch.randn(n, device='cuda', generator=g)
    dz_buf = torch.full((n + GUARD,), float('nan'), device='cuda')
    L.check(L.lib.vited_train_gelu_backward(_ptr(da), _ptr(z), _ptr(dz_buf), n, _stream()), 'train_gelu_backward')
    torch.cuda.synchronize()
    _assert_guard(a_buf, n, 'a')
    _assert_guard(dz_buf, n, 'dz')
    z64, da64 = z.double(), da.double()
    gelu = 0.5 * z64 * (1 + torch.erf(z64 / math.sqrt(2)))
    a = a_buf[:n].double()
    tol_a = _u16() * gelu.abs() + E32 * (2 * z64.abs() + gelu.abs()) + 2.0 ** -25
    err_a = ((a - gelu).abs() / tol_a).max().item()
    pdf = torch.exp(-0.5 * z64 * z64) / math.sqrt(2 * math.pi)
    dgelu = 0.5 * (1 + torch.erf(z64 / math.sqrt(2))) + z64 * pdf
    ref = da64 * dgelu
    dz = dz_buf[:n].double()
    tol_dz = da64.abs() * E32 * (4 + 5 * (z64 * pdf).abs() + 2 * dgelu.abs()) + E32 * ref.abs()
    err_dz = ((dz - ref).abs() / tol_dz).max().item()
    _report(f'gelu n {n} (errors / bound)', a=err_a, dz=err_dz, a_abs=(a - gelu).abs().max().item(),
            dz_abs=(dz - ref).abs().max().item())
    assert err_a <= 1.0, f'gelu forward exceeds its bound {err_a:.3g}x'
    assert err_dz <= 1.0, f'gelu backward exceeds its bound {err_dz:.3g}x'


# ---------------------------------------------------------------------------------------------------------------
# 4. bias-gradient column sums
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('N', [4, 384, 1152, 1540])
@pytest.mark.parametrize('R', [1, 7, 73800, 300001])
def test_colsum(R, N):
    """db[c] += alpha sum_r dy[r, c] against float64. Each thread sums rows r, r + step, ... (four at a time, then a
    remainder loop), eight row groups meet in shared memory, and one atomicAdd per column and row block lands on the
    prefill: |db - prefill - ref| <= (ceil(R / step) + gy + 12) 2^-24 (|prefill| + |alpha| sum_r |dy[r, c]|), with
    gy = min(ceil(R / 128), 592) row blocks and step = 8 gy, as the launcher picks them. Measured on a B200: at most
    0.18 of the bound (at R = 7), 3.4e-4 of it at R >= 73,800."""
    L = _lib()
    g = _gen(R + N)
    dy = torch.randn(R, N, device='cuda', generator=g)
    db_buf, db = _guarded(torch.randn(N, device='cuda', generator=g))
    pre = db.double()
    alpha = -0.7
    L.check(L.lib.vited_train_colsum(_ptr(dy), _ptr(db), R, N, alpha, _stream()), 'train_colsum')
    torch.cuda.synchronize()
    _assert_guard(db_buf, N, 'db')
    gy = min((R + 127) // 128, 148 * 4)
    depth = (R + 8 * gy - 1) // (8 * gy) + gy + 12
    ref = alpha * dy.double().sum(0)
    tol = depth * E32 * (pre.abs() + abs(alpha) * dy.double().abs().sum(0))
    err = ((db.double() - pre - ref).abs() / tol).max().item()
    _report(f'colsum R {R} N {N} (error / bound)', db=err)
    assert err <= 1.0, f'colsum exceeds its bound {err:.3g}x'


def test_colsum_rejects_bad_shapes_loudly():
    """The float4 loads need N % 4 == 0 and a 16-byte aligned dy: anything else is a non-zero status with a message
    and nothing written."""
    L = _lib()
    dy = torch.randn(9 * 64 + 4, device='cuda')
    db = torch.zeros(64, device='cuda')
    msg = _status_fails(L.lib.vited_train_colsum(_ptr(dy), _ptr(db), 8, 62, 1.0, _stream()), 'colsum N = 62')
    assert 'colsum' in msg
    misaligned = ctypes.c_void_p(dy.data_ptr() + 4)
    msg = _status_fails(L.lib.vited_train_colsum(misaligned, _ptr(db), 8, 64, 1.0, _stream()), 'colsum misaligned dy')
    assert 'colsum' in msg
    torch.cuda.synchronize()
    assert (db == 0).all()


# ---------------------------------------------------------------------------------------------------------------
# 5. transpose, cast, axpby16, axpy32: bit-exact
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('cfg', [
    # (R, C, ld_in, ld_out, scale, fp32 input)
    (1025, 384, 384, 1032, 1.0, False), (1025, 1152, 1152, 1032, 1024.0, True), (73, 45, 64, 80, 0.375, True),
    (33, 100, 100, 33, 1.0, True), (7, 31, 40, 8, -3.0, False), (1, 1, 1, 8, 1024.0, True), (64, 32, 33, 64, 1.0, True),
], ids=lambda c: 'x'.join(map(str, c)))
def test_transpose(cfg):
    """out [C, ld_out] 16-bit = scale * in[R, C]^T (fp32 or 16-bit input with row stride ld_in), rows R..ld_out-1 of
    the K dimension exactly 0: bit-identical to torch's fp32 multiply and round-to-nearest 16-bit conversion (with the
    kernels' fp16 saturation). The padding columns start as NaN; the rows past C stay NaN."""
    L = _lib()
    R, C, ld_in, ld_out, scale, f32 = cfg
    g = _gen(R * C)
    src = torch.randn(R, ld_in, device='cuda', generator=g) * 30.0
    if not f32:
        src = src.to(_act())
    out_buf = torch.full((C + GUARD, ld_out), float('nan'), dtype=_act(), device='cuda')
    L.check(L.lib.vited_train_transpose(_ptr(src), int(f32), ld_in, _ptr(out_buf), ld_out, R, C, scale, _stream()),
            'train_transpose')
    torch.cuda.synchronize()
    ref = _to16(src[:, :C].float().t() * scale)
    assert torch.equal(out_buf[:C, :R], ref), 'transpose is not bit-exact'
    assert (out_buf[:C, R:].float() == 0).all(), 'the padding rows of the K dimension must be exactly 0'
    _assert_guard(out_buf, C, 'transpose out')


def test_transpose_rejects_short_leading_dimensions():
    L = _lib()
    x = torch.zeros(8, 8, device='cuda')
    out = torch.zeros(8, 8, dtype=_act(), device='cuda')
    msg = _status_fails(L.lib.vited_train_transpose(_ptr(x), 1, 8, _ptr(out), 7, 8, 8, 1.0, _stream()), 'ld_out < R')
    assert 'transpose' in msg


@pytest.mark.parametrize('n', [0, 1, 1000, 1_234_567])
def test_cast_with_loss_scale(n):
    """out = 16-bit(in * scale), bit-identical to torch's fp32 multiply and round-to-nearest conversion. Values past
    the fp16 range saturate to +-65504 (fp16 builds), inf included: the cast feeds the 16-bit GEMM operands of the
    backward pass (loss-scaled dY, weights), and with a fixed loss scale and no step skipping an inf operand would turn
    whole GEMM rows into inf / NaN (inf * 0 in the zero padding of K) and poison every gradient it reaches; a saturated
    value keeps the step finite, the same policy test_fp16_results_saturate_instead_of_overflowing pins for the GEMM.
    bf16 builds have the fp32 range: there the result is torch's conversion, inf stays inf."""
    L = _lib()
    g = _gen(n + 5)
    x = torch.randn(max(n, 1), device='cuda', generator=g)[:n] * 20.0
    if n >= 1000:
        # * 1024: +-71680, +-1.0e6, 65519 (rounds to 65504) and 65520 (the fp16 rounding midpoint to inf), and two
        # values whose product overflows fp32 to +-inf
        x[:8] = torch.tensor([70.0, -70.0, 1000.0, -1000.0, 65519.0 / 1024, 65520.0 / 1024, 3e38, -3e38],
                             device='cuda')
    scale = 1024.0
    out_buf = torch.full((n + GUARD,), float('nan'), dtype=_act(), device='cuda')
    L.check(L.lib.vited_train_cast(_ptr(x), _ptr(out_buf), n, scale, _stream()), 'train_cast')
    torch.cuda.synchronize()
    ref = _to16(x * scale)
    assert torch.equal(out_buf[:n], ref), 'cast is not bit-exact'
    _assert_guard(out_buf, n, 'cast out')
    if n >= 1000 and _act() == torch.float16:
        assert (out_buf[:8].float().abs() == 65504.0).all(), 'fp16 values out of range must saturate'
        assert torch.isfinite(out_buf[:n].float()).all()


@pytest.mark.parametrize('n', [0, 1, 1000, 1_234_567])
@pytest.mark.parametrize('ab', [(1.0 / 1024, 1.0), (1.0, 0.0), (0.75, 1.5), (-1.5, 0.0)], ids=lambda a: f'{a[0]}_{a[1]}')
def test_axpby16(n, ab):
    """y = alpha * x16 + beta * y (fp32 y): bit-identical to torch's fp32 arithmetic. The kernel computes
    fma(alpha, x, beta * y); alpha has few significand bits here, as train.py's alpha (1 / loss scale, 1) has, so
    alpha * x is exact and the FMA rounds like torch's separate add. With beta = 0, y is not read: a NaN already in y
    does not reach the result."""
    L = _lib()
    alpha, beta = ab
    g = _gen(n + 11)
    x = (torch.randn(max(n, 1), device='cuda', generator=g)[:n] * 8.0).to(_act())
    y_buf, y = _guarded(torch.randn(n, device='cuda', generator=g) * 3.0)
    if beta == 0.0 and n:
        y[::7] = float('nan')
    pre = y.clone()
    L.check(L.lib.vited_train_axpby16(_ptr(x), _ptr(y), n, alpha, beta, _stream()), 'train_axpby16')
    torch.cuda.synchronize()
    ref = alpha * x.float() if beta == 0.0 else alpha * x.float() + beta * pre
    assert torch.equal(y, ref), 'axpby16 is not bit-exact'
    _assert_guard(y_buf, n, 'axpby16 y')


@pytest.mark.parametrize('n', [0, 1, 1000, 1_234_567])
@pytest.mark.parametrize('alpha', [1.0, -0.5, 1.0 / 1024])
def test_axpy32(n, alpha):
    """y += alpha * x (fp32): the kernel's fma(alpha, x, y) is bit-identical to torch's y + alpha * x for the
    power-of-two alphas used here (the product is exact; train.py passes 1)."""
    L = _lib()
    g = _gen(n + 13)
    x = torch.randn(max(n, 1), device='cuda', generator=g)[:n]
    y_buf, y = _guarded(torch.randn(n, device='cuda', generator=g))
    pre = y.clone()
    L.check(L.lib.vited_train_axpy32(_ptr(x), _ptr(y), n, alpha, _stream()), 'train_axpy32')
    torch.cuda.synchronize()
    assert torch.equal(y, pre + alpha * x), 'axpy32 is not bit-exact'
    _assert_guard(y_buf, n, 'axpy32 y')


# ---------------------------------------------------------------------------------------------------------------
# 6. row gather / scatter-add, with the exact calls train.py makes
# ---------------------------------------------------------------------------------------------------------------
def _hisfrag_indices(B=24, writers=8):
    from vited_b200 import train
    targets = torch.arange(B) // (B // writers)
    groups, _ = train.prepare_pairs(targets, torch.Generator().manual_seed(1))
    P = groups.shape[0]
    g0 = groups[:, 0].to(device='cuda', dtype=torch.int32).contiguous()
    g1 = groups[:, 1].to(device='cuda', dtype=torch.int32).contiguous()
    zeros = torch.zeros(max(B, P), dtype=torch.int32, device='cuda')
    arange_p = torch.arange(P, dtype=torch.int32, device='cuda')
    return B, P, g0, g1, zeros, arange_p


def _block_rows(idx, n_blocks, rows_per, stride, off, indexed):
    blk = idx[:n_blocks].long() if indexed else torch.arange(n_blocks, device='cuda')
    return (blk[:, None] * stride + off + torch.arange(rows_per, device='cuda')[None, :]).reshape(-1)


def test_gather_rows_train_calls():
    """out block b, row t = in block idx[b], row t (+= when accumulate): the six gathers of train.py's forward at the
    Hisfrag20 shape (24 images of 1,024 tokens, 72 pairs of 1,025). Exact: a copy or one fp32 add. Rows of the output
    that no block names keep their prefill bit for bit."""
    L = _lib()
    B, P, g0, g1, zeros, arange_p = _hisfrag_indices()
    assert g0.unique().numel() < P and g1.unique().numel() < P, 'the pair indices must repeat items'
    ne, nd, D = 1024, 1025, 384
    g = _gen(5)
    pos = torch.randn(nd, D, device='cuda', generator=g)
    cls = torch.randn(1, D, device='cuda', generator=g)
    tok = torch.randn(B * ne, D, device='cuda', generator=g)
    enc = torch.randn(B * ne, D, device='cuda', generator=g)
    x_pair = torch.randn(P * nd, D, device='cuda', generator=g)
    calls = [
        # (what, in, idx, n_blocks, rows_per, in_stride, in_off, out rows, out_stride, out_off, accumulate)
        ('encoder input = pos[1:]', pos, zeros, B, ne, nd, 1, B * ne, ne, 0, False),
        ('decoder input = pos', pos, zeros, P, nd, nd, 0, P * nd, nd, 0, False),
        ('decoder cls rows += cls', cls, zeros, P, 1, 1, 0, P * nd, nd, 0, True),
        ('decoder rows 1.. += tokens[g0]', tok, g0, P, ne, ne, 0, P * nd, nd, 1, True),
        ('context = encoder out[g1]', enc, g1, P, ne, ne, 0, P * ne, ne, 0, False),
        ('class-token rows', x_pair, arange_p, P, 1, nd, 0, P, 1, 0, False),
    ]
    for what, src, idx, nb, rp, ist, ioff, nrows, ost, ooff, acc in calls:
        buf, out = _guarded(torch.randn(nrows, D, device='cuda', generator=g))
        pre = out.clone()
        L.check(L.lib.vited_train_gather_rows(_ptr(src), _ptr(idx), _ptr(out), nb, rp, ist, ioff, ost, ooff, D, int(acc),
                                              _stream()), 'train_gather_rows')
        torch.cuda.synchronize()
        src_rows = _block_rows(idx, nb, rp, ist, ioff, True)
        dst_rows = _block_rows(idx, nb, rp, ost, ooff, False)
        ref = pre.clone()
        ref[dst_rows] = pre[dst_rows] + src[src_rows] if acc else src[src_rows]
        assert torch.equal(out, ref), f'{what}: gather is not exact (or touched rows it does not name)'
        _assert_guard(buf, nrows, what)


def test_scatter_add_rows_train_calls():
    """dst block idx[b], row t += alpha * src block b, row t (atomicAdd): the six scatter-adds of train.py's
    backward at the Hisfrag20 shape, against float64 index_add_. A destination row that m blocks name is a sum of m
    fp32 atomic adds in any order onto the prefill: |dst - prefill - ref| <= (m + 2) 2^-24 (|prefill| + sum |alpha
    src|). The all-zeros index adds every pair into pos_embed (m = 72); g0 / g1 repeat items. Rows that no block names
    keep their prefill bit for bit. Measured on a B200: at most 0.50 of the bound."""
    L = _lib()
    B, P, g0, g1, zeros, arange_p = _hisfrag_indices()
    ne, nd, D = 1024, 1025, 384
    g = _gen(6)
    inv = 1.0 / 1024
    dxc = torch.randn(P, D, device='cuda', generator=g)
    dx_pair = torch.randn(P * nd, D, device='cuda', generator=g)
    dctx = torch.randn(P * ne, D, device='cuda', generator=g)
    dx_enc = torch.randn(B * ne, D, device='cuda', generator=g)
    calls = [
        # (what, src, idx, n_blocks, rows_per, src_stride, src_off, dst rows, dst_stride, dst_off, alpha)
        ('class-token rows of dx', dxc, arange_p, P, 1, 1, 0, P * nd, nd, 0, 1.0),
        ('pos_embed from the pairs', dx_pair, zeros, P, nd, nd, 0, nd, nd, 0, inv),
        ('cls_token', dx_pair, zeros, P, 1, nd, 0, 1, 1, 0, inv),
        ('tokens[g0]', dx_pair, g0, P, ne, nd, 1, B * ne, ne, 0, 1.0),
        ('encoder out[g1]', dctx, g1, P, ne, ne, 0, B * ne, ne, 0, 1.0),
        ('pos_embed[1:] from the encoder', dx_enc, zeros, B, ne, ne, 0, nd, nd, 1, inv),
    ]
    worst = 0.0
    for what, src, idx, nb, rp, sst, soff, nrows, dst_st, doff, alpha in calls:
        buf, dst = _guarded(torch.randn(nrows, D, device='cuda', generator=g))
        pre = dst.clone()
        L.check(L.lib.vited_train_scatter_add_rows(_ptr(src), _ptr(idx), _ptr(dst), nb, rp, sst, soff, dst_st, doff, D,
                                                   alpha, _stream()), 'train_scatter_add_rows')
        torch.cuda.synchronize()
        src_rows = _block_rows(idx, nb, rp, sst, soff, False)
        dst_rows = _block_rows(idx, nb, rp, dst_st, doff, True)
        ref = torch.zeros(nrows, D, dtype=torch.float64, device='cuda').index_add_(0, dst_rows,
                                                                                   alpha * src[src_rows].double())
        mag = torch.zeros_like(ref).index_add_(0, dst_rows, (alpha * src[src_rows].double()).abs())
        cnt = torch.zeros(nrows, dtype=torch.float64, device='cuda').index_add_(
            0, dst_rows, torch.ones(dst_rows.numel(), dtype=torch.float64, device='cuda'))
        tol = (cnt[:, None] + 2) * E32 * (pre.double().abs() + mag)
        err = ((dst.double() - pre.double() - ref).abs() / tol)
        named = cnt > 0
        assert torch.equal(dst[~named], pre[~named]), f'{what}: rows that no block names changed'
        e = err[named].max().item()
        worst = max(worst, e)
        assert e <= 1.0, f'{what}: scatter-add exceeds its bound {e:.3g}x'
        _assert_guard(buf, nrows, what)
    _report('scatter_add (error / bound)', worst=worst)


# ---------------------------------------------------------------------------------------------------------------
# 7. BCE-with-logits
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('n', [1, 72, 257, 5000])
def test_bce_logits(n):
    """loss = mean BCE-with-logits, dlogits = (sigmoid(x) - y) * grad_scale / n, against float64 torch. One 256-thread
    block: 257 and 5,000 elements take the per-thread loop. Logits include 0, +-30 and +-100; labels are 0 / 1 and
    fractional.

    Bounds: each term max(x, 0) - x y + log1p(exp(-|x|)) is within 2^-24 4 (|x| + 1) of exact; summed in per-thread,
    warp and block order: |loss - ref| <= 2^-24 ((ceil(n / 256) + 16) sum term + 4 sum(|x| + 1)) / n. sigmoid = 1 / (1 +
    exp(-x)) is within 5 ulp, then the difference, the scale and the division round: |dlogit - ref| <= grad_scale / n
    2^-24 (5 sigmoid + 3 |sigmoid - y|). Measured on a B200, as a fraction of the bounds: loss 0.027, dlogits 0.48."""
    L = _lib()
    g = _gen(n + 17)
    x = torch.randn(n, device='cuda', generator=g) * 4.0
    special = torch.tensor([0.0, 30.0, -30.0, 100.0, -100.0], device='cuda')
    x[:min(n, 5)] = special[:min(n, 5)]
    y = (torch.rand(n, device='cuda', generator=g) > 0.5).float()
    y[1::3] = torch.rand(y[1::3].shape, device='cuda', generator=g)          # fractional labels
    gs = 1024.0
    loss_buf = torch.full((1 + GUARD,), float('nan'), device='cuda')
    dl_buf = torch.full((n + GUARD,), float('nan'), device='cuda')
    L.check(L.lib.vited_train_bce_logits(_ptr(x), _ptr(y), n, _ptr(loss_buf), _ptr(dl_buf), gs, _stream()),
            'train_bce_logits')
    torch.cuda.synchronize()
    _assert_guard(loss_buf, 1, 'loss')
    _assert_guard(dl_buf, n, 'dlogits')
    x64, y64 = x.double(), y.double()
    terms = x64.clamp_min(0) - x64 * y64 + torch.log1p(torch.exp(-x64.abs()))
    ref_loss = torch.nn.functional.binary_cross_entropy_with_logits(x64, y64)
    loss = loss_buf[0].double()
    assert torch.isfinite(loss)
    tol_loss = E32 * ((math.ceil(n / 256) + 16) * terms.sum() + 4 * (x64.abs() + 1).sum()) / n
    sig = torch.sigmoid(x64)
    ref_dl = (sig - y64) * gs / n
    tol_dl = gs / n * E32 * (5 * sig + 3 * (sig - y64).abs()) + 1e-38
    err_loss = ((loss - ref_loss).abs() / tol_loss).item()
    err_dl = ((dl_buf[:n].double() - ref_dl).abs() / tol_dl).max().item()
    _report(f'bce n {n} (errors / bound)', loss=err_loss, dlogits=err_dl)
    assert err_loss <= 1.0, f'loss {loss.item()} vs {ref_loss.item()}'
    assert err_dl <= 1.0, f'dlogits exceed their bound {err_dl:.3g}x'


def test_bce_rejects_an_empty_batch():
    L = _lib()
    buf = torch.zeros(4, device='cuda')
    msg = _status_fails(L.lib.vited_train_bce_logits(_ptr(buf), _ptr(buf), 0, _ptr(buf), _ptr(buf), 1.0, _stream()),
                        'bce n = 0')
    assert 'bce' in msg


# ---------------------------------------------------------------------------------------------------------------
# 8. one training step at the Hisfrag20 token count
# ---------------------------------------------------------------------------------------------------------------
# every parameter gradient, relative L2 error against float64 autograd, in units of u: measured 7.4u (fp16, 0.36 %)
# and 18.4u (bf16, 7.2 %), both on bias / LayerNorm-bias gradients, sums over all rows of a 16-bit-rounded gradient
STEP_REL_L2 = {torch.float16: 16, torch.bfloat16: 32}
STEP_ELEM = 8       # qkv / kv / proj weight gradients, element by element, relative to each tensor's max, in units of
                    # u: measured 2.3u (fp16) and 3.5u (bf16)


def test_train_step_at_hisfrag20_token_count():
    """train.train_step on a Hisfrag20-shaped model cut to depth = c_depth = 1 (img 512, patch 16, embed 384, 6
    heads: 1,024 encoder and 1,025 decoder tokens), 6 images of two writers (15 pairs), against float64 autograd of the
    oracle on the same state_dict, samples, targets and randperm seed. Every gradient tensor by relative L2; the
    qkv, kv and proj weight gradients also element by element (relative to each tensor's max). The error comes from
    the 16-bit GEMM and attention operands: bounds in units of u (STEP_REL_L2, STEP_ELEM). Measured on a B200 (fp16):
    every gradient within 0.36 % relative L2 (the weight gradients within 0.20 %), qkv / kv / proj weight gradients
    within 1.1e-3 of their max, loss within 2e-5; the float64 oracle takes a few seconds on the host."""
    import vited_b200
    from vited_b200 import synthetic, train
    from oracle import vited_oracle as orc
    from tests import helpers
    _, kw = helpers.load_model_case('hisfrag20_patch16_512')
    kw = dict(kw, depth=1, c_depth=1)
    model, sd = helpers.make_gpu_model(kw, 31)
    targets = [0, 0, 0, 1, 1, 1]
    samples = synthetic.synthetic_images(len(targets), kw['img_size'], seed=131)
    perm_seed = 9
    torch.manual_seed(perm_seed)
    loss, logits, groups, labels = train.train_step(model, samples.cuda(), targets)
    torch.cuda.synchronize()
    assert groups.shape[0] == 15
    o_loss, o_logits, o_groups, o_labels, o_grads = orc.train_step({k: v.double() for k, v in sd.items()},
                                                                   kw['num_heads'], samples.double(), targets, perm_seed)
    assert torch.equal(groups, o_groups) and torch.equal(labels, o_labels)
    u = _u16()
    rel_l2, elem = {}, {}
    for k, p in model.named_parameters():
        got, want = p.grad.detach().cpu().double(), o_grads[k].double()
        assert torch.isfinite(got).all(), k
        assert want.norm() > 0, k
        rel_l2[k] = float((got - want).norm() / want.norm())
        if k.endswith(('qkv.weight', 'kv.weight', 'proj.weight')) and not k.startswith('patch_embed'):
            elem[k] = float((got - want).abs().max() / want.abs().max())
    worst_key = max(rel_l2, key=rel_l2.get)
    worst = rel_l2[worst_key]
    _report('train step Hisfrag20 tokens', loss=abs(loss.item() - o_loss.item()), worst_rel_l2=worst,
            worst_rel_l2_in_u=worst / u, worst_elem=max(elem.values()), worst_elem_in_u=max(elem.values()) / u)
    print(f'worst relative L2: {worst_key}; relative L2: {rel_l2}; element errors: {elem}')
    assert len(elem) == 6
    for k, e in rel_l2.items():
        assert e <= STEP_REL_L2[_act()] * u, f'{k}: relative L2 error {e:.3g}'
    for k, e in elem.items():
        assert e <= STEP_ELEM * u, f'{k}: element error {e:.3g} of the max'
    assert abs(loss.item() - o_loss.item()) <= 4 * u * max(1.0, o_loss.item())
    assert (logits.cpu().double() - o_logits).abs().max().item() <= 64 * u * max(1.0, o_logits.abs().max().item())
