"""GPU: the cross-attention projection + residual + norm2 fused in front of the MLP sub-block (vited_op_cproj_mlp_resid_ln,
mlp_ln.cu with its prologue), against fp32 torch on the same 16-bit operands and against the two kernels it replaces
(gemm_resid_ln for the projection, then mlp_resid_ln)."""
import ctypes
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

D = 384


def _lib():
    from vited_b200 import _lib
    return _lib


def _act():
    return _lib().act_dtype()


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _operands(M, HID, big):
    g = torch.Generator(device='cuda').manual_seed(M + HID + (7 if big else 0))
    r = lambda *s: torch.randn(*s, device='cuda', generator=g)
    o = r(M, D).to(_act())
    Wp = (r(D, D) / math.sqrt(D)).to(_act())
    bp = r(D)
    W1 = (r(HID, D) / math.sqrt(D)).to(_act())
    b1 = 0.5 * r(HID)
    W2 = (r(D, HID) / math.sqrt(HID)).to(_act())
    b2 = r(D)
    if big:   # |x| ~ 100: fc2 accumulates onto 2 x_mid, whose fp32 ulp is ~1e-5
        x = 100.0 + r(M, D) * 2
    else:     # rows with a large common offset exercise the shifted variance of both LayerNorms
        x = r(M, D) * 2 + r(M, 1) * 5
    ln2 = (1 + 0.1 * r(D), 0.1 * r(D))
    ln1 = (1 + 0.1 * r(D), 0.1 * r(D))
    return o, Wp, bp, x, ln2, W1, b1, W2, b2, ln1


def _fused(M, HID, o, Wp, bp, x, ln2, W1, b1, W2, b2, ln1):
    L = _lib()
    h = torch.full((M, D), float('nan'), dtype=_act(), device='cuda')
    L.check(L.lib.vited_op_cproj_mlp_resid_ln(_ptr(o), _ptr(Wp), _ptr(bp), _ptr(x), _ptr(ln2[0]), _ptr(ln2[1]), _ptr(W1),
                                              _ptr(b1), _ptr(W2), _ptr(b2), _ptr(ln1[0]), _ptr(ln1[1]), _ptr(h), M, D,
                                              HID, 1e-6, _stream()), 'op_cproj_mlp_resid_ln')
    torch.cuda.synchronize()
    return h


@pytest.mark.parametrize('big', [False, True], ids=['offset_rows', 'abs100'])
@pytest.mark.parametrize('shape', [(256, 1536), (33333, 1536), (70000, 1536), (262144 + 77, 1536), (1, 1536),
                                   (100, 1536), (300, 64), (40000, 192)], ids=lambda s: 'x'.join(map(str, s)))
def test_cproj_mlp_resid_ln_fused(shape, big):
    """x_mid = x + o Wp^T + bp; h2 = norm2(x_mid); x = x_mid + fc2(GELU(fc1(h2))) + b2; h = norm1'(x), with h2 and the
    hidden activations rounded to 16 bits where the kernel rounds them. x holds the final rows (x_mid is never
    written to it) and o is left as it was."""
    M, HID = shape
    o, Wp, bp, x, ln2, W1, b1, W2, b2, ln1 = _operands(M, HID, big)
    o_in = o.clone()
    x_mid = x + o.float() @ Wp.float().t() + bp
    h2 = torch.nn.functional.layer_norm(x_mid, (D,), *ln2, 1e-6).to(_act()).float()
    mlp = torch.nn.functional.gelu(h2 @ W1.float().t() + b1).to(_act()).float() @ W2.float().t() + b2
    x_ref = x_mid + mlp
    h_ref = torch.nn.functional.layer_norm(x_ref, (D,), *ln1, 1e-6)
    del h2
    h = _fused(M, HID, o, Wp, bp, x, ln2, W1, b1, W2, b2, ln1)
    assert torch.equal(o, o_in)
    assert torch.isfinite(h.float()).all() and torch.isfinite(x).all()
    r16 = 1.0 if _act() == torch.bfloat16 else 0.2
    # the MLP term as in test_mlp_resid_ln_fused (a hidden value next to a 16-bit rounding boundary may round the other
    # way, over K = hidden), plus the fp32 accumulation onto 2 x_mid: one ulp of |x| per MMA k-step at most
    tol_x = (2e-3 if _act() == torch.float16 else 1.5e-2) * max(1.0, mlp.abs().max().item()) + \
        1.2e-7 * (HID / 16) * x_ref.abs().max().item()
    err_x = (x - x_ref).abs().max().item()
    assert err_x < tol_x, (err_x, tol_x)
    # h2 itself is a 16-bit rounding: its error reaches h through the MLP
    assert (h.float() - h_ref).abs().max().item() <= (1e-2 * h_ref.abs().max().item() + 4e-3) * r16 + \
        2 * tol_x / x_ref.std(dim=1).min().item()


@pytest.mark.parametrize('big', [False, True], ids=['offset_rows', 'abs100'])
@pytest.mark.parametrize('M', [70000, 262144 + 77])
def test_cproj_mlp_resid_ln_matches_the_unfused_pair(M, big):
    """The fused launch against gemm_resid_ln (projection + residual + norm2) followed by mlp_resid_ln on the same
    operands: h2 is computed operation for operation as gemm_resid_ln computes it, so the only difference is that x_mid
    enters the fp32 sum of fc2 on the tensor core instead of after it."""
    HID = 1536
    L = _lib()
    o, Wp, bp, x, ln2, W1, b1, W2, b2, ln1 = _operands(M, HID, big)
    x_pair = x.clone()
    h_pair = torch.empty(M, D, dtype=_act(), device='cuda')
    L.check(L.lib.vited_op_gemm_resid_ln(_ptr(o), _ptr(Wp), _ptr(bp), _ptr(x_pair), _ptr(ln2[0]), _ptr(ln2[1]),
                                         _ptr(h_pair), M, D, D, 1e-6, _stream()), 'op_gemm_resid_ln')
    L.check(L.lib.vited_op_mlp_resid_ln(_ptr(h_pair), _ptr(W1), _ptr(b1), _ptr(W2), _ptr(b2), _ptr(x_pair), _ptr(ln1[0]),
                                        _ptr(ln1[1]), _ptr(h_pair), M, D, HID, 1e-6, _stream()), 'op_mlp_resid_ln')
    h = _fused(M, HID, o, Wp, bp, x, ln2, W1, b1, W2, b2, ln1)
    # fp32 rounding of one sum in a different order: a few ulps of |x| per MMA k-step at most
    tol_x = 1.2e-7 * (HID / 16) * x_pair.abs().max().item() + 1e-6
    err_x = (x - x_pair).abs().max().item()
    assert err_x < tol_x, (err_x, tol_x)
    # the normalised rows then differ by at most one 16-bit rounding step
    step = 2.0 ** (-7 if _act() == torch.bfloat16 else -10)
    err_h = (h.float() - h_pair.float()).abs().max().item()
    assert err_h <= 2 * step * h_pair.float().abs().max().item(), err_h
