"""GPU: the scoring-path kernels one by one (the fused LayerNorm kernels, the GEMM, the three attention kernels, the
class-token-only attention of the pruned last decoder layer, and the final LayerNorm + head) against a float64 torch
computation of the same operation on the same 16-bit-rounded operands, rounding to 16 bits where the kernel rounds.

Every output buffer carries NaN sentinel rows past its end, and wherever the kernel must not write; in-place outputs
(the residual stream ``x`` of the fused kernels) are checked as ``result - prefill``.

Tolerances are per element and written in units of u, the unit roundoff of the 16-bit type the library was built with
(2^-11 fp16, 2^-8 for -DVITED_ACT_BF16=1 builds), and of 2^-24 for fp32 arithmetic. Each test's docstring derives its
bound from the roundings the kernel does and quotes the largest ratio error / bound measured on a B200 (each test
prints it with -s). Besides random operands, inputs are built to expose specific bugs: rows whose
LayerNorm output is exactly +-1, and keys that dominate a softmax row by ~70 nats."""
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
N_ACC = 32          # longest chain of fp32 additions in any row sum of the LayerNorm kernels (29 in resid_ln at D = 768)
GELU_ERR = 1e-4     # |GELU epilogue - exact erf GELU| (test_gpu_kernels.py::test_gelu_epilogue_accuracy)
EPS_EXP = 8.6e-5    # relative error of the exponentials (the ex2_poly2 polynomial of attention_tc.cu; MUFU.EX2 is finer)
RSQRT_ERR = 2.0 ** -21   # relative error of rsqrtf (MUFU.RSQ)
LN_EPS = 1e-6
D = 384             # embed_dim of both models (the only width the fused kernels take)
CHUNK = 65536       # rows per float64 reference slice


def _lib():
    from vited_b200 import _lib
    return _lib


def _act():
    return _lib().act_dtype()


def _u16():
    """unit roundoff of the 16-bit activation type: 2^-8 (bf16) or 2^-11 (fp16)"""
    return 2.0 ** -8 if _act() == torch.bfloat16 else 2.0 ** -11


def _tiny16():
    """largest rounding error of a 16-bit result below the normal range (fp16 subnormal spacing / 2; bf16 has none here)"""
    return 2.0 ** -25 if _act() == torch.float16 else 2.0 ** -134


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _gen(seed):
    return torch.Generator(device='cuda').manual_seed(seed)


def _nan_buf(rows, cols, dtype):
    """(buffer, view): a NaN-filled buffer of rows + GUARD rows; the view is the first ``rows``"""
    buf = torch.full((rows + GUARD, cols), float('nan'), dtype=dtype, device='cuda')
    return buf, buf[:rows]


def _assert_guard(buf, n, what):
    assert torch.isnan(buf[n:].float()).all(), f'{what}: the rows past the end of the output were written'


def _report(name, **vals):
    print(f'[{_act()}] {name}: ' + ', '.join(f'{k} {v:.3g}' for k, v in vals.items()))


def _check(err, bound, what):
    """err <= bound element by element; returns the largest ratio err / bound (the figure quoted in docstrings)"""
    bad = ~(err <= bound)
    if bad.any():
        i = bad.nonzero()[0].tolist()
        raise AssertionError(f'{what}: {int(bad.sum())} / {bad.numel()} elements over the bound; first {i}: '
                             f'err {float(err[tuple(i)]):.4g} > bound {float(bound[tuple(i)]):.4g}; '
                             f'max err {float(err.max()):.4g}')
    return float((err / bound).max())


# ---------------------------------------------------------------------------------------------------------------
# 16-bit rounding helpers (float64 in, float64 out)
# ---------------------------------------------------------------------------------------------------------------
def _r16(x):
    return x.to(_act()).double()


def _step(r):
    """spacing of the 16-bit grid just above |r| (r on the grid): 2u * 2^floor(log2|r|), at least the subnormal step"""
    _, e = torch.frexp(r)
    sp = torch.ldexp(torch.full_like(r, _u16()), e).clamp_min(2 * _tiny16())
    return torch.where(r == 0, torch.full_like(r, 2 * _tiny16()), sp)


def _flips(g, eps):
    """Largest change of round16(g) when g is perturbed by at most eps (element-wise): zero unless a rounding boundary
    lies within eps of g, else one grid step per boundary crossed. The step below a power of two is half the step above."""
    r = _r16(g)
    sp = _step(r)
    m, _ = torch.frexp(r)
    below = torch.where(m.abs() == 0.5, sp / 2, sp)
    dist = below / 2 - (g - r).abs()          # distance to the nearest boundary (conservative at powers of two)
    crossings = 1 + torch.floor(eps / below)
    return torch.where(dist <= eps, crossings * sp, torch.zeros_like(g))


# ---------------------------------------------------------------------------------------------------------------
# 1. LayerNorm-carrying kernels: resid_ln (rowops.cu), gemm_resid_ln (gemm_ln.cu), mlp_resid_ln and its cross-projection
#    prologue (mlp_ln.cu)
# ---------------------------------------------------------------------------------------------------------------
def _ln64(v, w, b):
    mean = v.mean(1, keepdim=True)
    c = v - mean
    rstd = 1.0 / torch.sqrt((c * c).mean(1, keepdim=True) + LN_EPS)
    xhat = c * rstd
    return xhat * w + b, xhat, rstd


def _ln_terms(v, e, w, b, pivots):
    """fp32 error terms of h = LayerNorm(v) * w + b before its 16-bit rounding, element by element:
      * the statistics: the mean is a sum of D fp32 values along chains of at most N_ACC additions, so
        |d mean| <= N_ACC 2^-24 mean|v|; the variance is a sum of squares about a pivot p (the group's first element in
        the tcgen05 epilogues, the mean in rowops.cu), relative error <= 2 N_ACC 2^-24 sum (v-p)^2 / sum (v-mean)^2, and
        rsqrtf adds 2^-21: |d rstd| / rstd <= N_ACC 2^-24 ratio + 2^-21;
      * the four fp32 operations (v - mean) * rstd * w + b: 4 * 2^-24 (|xhat w| + |b|);
      * the propagated error e of the row v itself (measured: the kernel's own x against the reference), to first order
        in e / std: |w| rstd (|e_i| + mean|e| + |xhat_i| mean|xhat e|)."""
    w, b = w.double(), b.double()
    h, xhat, rstd = _ln64(v, w, b)
    c2 = ((v - v.mean(1, keepdim=True)) ** 2).sum(1, keepdim=True)
    if pivots is None:
        ratio = torch.ones_like(c2)
    else:
        ratio = torch.stack([((v - v[:, p:p + 1]) ** 2).sum(1, keepdim=True) for p in pivots]).amax(0) / c2
    dmean = N_ACC * E32 * v.abs().mean(1, keepdim=True)
    drel = N_ACC * E32 * ratio + RSQRT_ERR
    aw = w.abs()
    t = rstd * aw * dmean + (xhat * w).abs() * drel + 4 * E32 * ((xhat * w).abs() + b.abs())
    if e is not None:
        ea = e.abs()
        t = t + 1.01 * rstd * aw * (ea + ea.mean(1, keepdim=True) + xhat.abs() * (xhat.abs() * ea).mean(1, keepdim=True))
    return h, t


def _h_bound(h_ref, terms):
    """one 16-bit rounding of the kernel's fp32 value, which lies within ``terms`` of h_ref"""
    return _u16() * h_ref.abs() + (1 + _u16()) * terms + _tiny16()


def _rows(M, width, kind, g):
    """fp32 residual rows: 'offset' = N(0, 2^2) + a per-row common offset N(0, 5^2) (the shifted statistics);
    'abs100' = 100 + N(0, 2^2) (the fp32 ulp of x is 2^-17)"""
    if kind == 'abs100':
        return 100.0 + 2 * torch.randn(M, width, device='cuda', generator=g)
    return 2 * torch.randn(M, width, device='cuda', generator=g) + 5 * torch.randn(M, 1, device='cuda', generator=g)


def _ln_params(width, g):
    return 1 + 0.1 * torch.randn(width, device='cuda', generator=g), 0.1 * torch.randn(width, device='cuda', generator=g)


def _check_ln_out(name, x_in, x_out, dx_ref, dx_bound, h, lw, lb, pivots):
    """x: (result - prefill) against the reference sub-block output within dx_bound; h: against float64 LayerNorm of
    the reference row within _h_bound, carrying the measured error of x. Row slices keep the float64 work bounded."""
    M = x_in.shape[0]
    worst_x = worst_h = 0.0
    for r0 in range(0, M, CHUNK):
        sl = slice(r0, min(M, r0 + CHUNK))
        xi = x_in[sl].double()
        dx = dx_ref(sl)
        e = x_out[sl].double() - xi - dx
        worst_x = max(worst_x, _check(e.abs(), dx_bound(sl, xi), f'{name}: x - prefill, rows {r0}+'))
        h_ref, terms = _ln_terms(xi + dx, e, lw, lb, pivots)
        worst_h = max(worst_h, _check((h[sl].double() - h_ref).abs(), _h_bound(h_ref, terms), f'{name}: h, rows {r0}+'))
    _report(name, x_err_over_bound=worst_x, h_err_over_bound=worst_h)


LN_KINDS = ['offset', 'abs100']


@pytest.mark.parametrize('kind', LN_KINDS)
@pytest.mark.parametrize('has_cls', [0, 1])
@pytest.mark.parametrize('width', [384, 768, 32, 96])
def test_resid_ln_float64(width, has_cls, kind):
    """x += delta; h = LayerNorm(x) (rowops.cu: the unrolled kernel at D = 384 / 768, the generic one at 32 / 96).
    x: one fp32 addition, |err| <= 2^-24 |x + delta|. h: _h_bound (one 16-bit rounding + the fp32 statistics, two-pass
    here so the pivot ratio is 1). In the fp16 build the bound is u |h| + O(1e-5), below the 1.3e-3 relative shift of a
    variance divided by D - 1. Measured on a B200 (1,000 W), largest err / bound, fp16 / bf16 build:
    x 1.0 / 1.0 (the bound is one fp32 rounding), h 0.99 / 0.995."""
    L = _lib()
    n_seq, n_patch = 37, 9
    rows = n_seq * n_patch + (n_seq if has_cls else 0)
    g = _gen(width * 4 + has_cls * 2 + LN_KINDS.index(kind))
    x_in = _rows(rows, width, kind, g)
    delta = torch.randn(rows, width, device='cuda', generator=g).to(_act())
    lw, lb = _ln_params(width, g)
    xbuf, x = _nan_buf(rows, width, torch.float32)
    x.copy_(x_in)
    hbuf, h = _nan_buf(rows, width, _act())
    L.check(L.lib.vited_op_resid_ln(_ptr(x), _ptr(delta), _ptr(lw), _ptr(lb), _ptr(h), n_seq, n_patch, has_cls, width,
                                    LN_EPS, _stream()), 'op_resid_ln')
    torch.cuda.synchronize()
    _assert_guard(xbuf, rows, 'x')
    _assert_guard(hbuf, rows, 'h')
    _check_ln_out(f'resid_ln D={width}', x_in, x, lambda sl: delta[sl].double(),
                  lambda sl, xi: E32 * (xi + delta[sl].double()).abs(), h, lw, lb, None)


GEMM_LN_SHAPES = [(256, 384), (70000, 384), (33333, 1536), (1, 384), (300, 64), (40000, 192)]
PIVOTS = [0, 96, 192, 288]   # first column of every column group of the two epilogue forms (2 x 192, 4 x 96)


def _epi_variant(epi_warps, monkeypatch):
    """The 16-warp (four 96-column groups) epilogue form exists in -DVITED_EXPERIMENTAL builds only."""
    if epi_warps == '16' and 'experimental' not in os.environ.get('VITED_LIB', ''):
        pytest.skip('16 epilogue warps: experimental build only (VITED_LIB=tools/bin/experimental/libvited_b200.so)')
    monkeypatch.setenv('VITED_EPI_WARPS', epi_warps)


@pytest.mark.parametrize('kind', LN_KINDS)
@pytest.mark.parametrize('shape', GEMM_LN_SHAPES, ids=lambda s: 'x'.join(map(str, s)))
def test_gemm_resid_ln_float64(shape, kind):
    """x += A W^T + b; h = LayerNorm(x) (gemm_ln.cu). x - prefill: the tensor-core fp32 accumulation over K plus the
    additions of b and x, |err| <= (K + 3) 2^-24 (sum_k |a_k w_k| + |b| + |x|). h: _h_bound with the Chan-combined
    statistics of the column groups (pivot ratio over the groups' first elements).
    Measured on a B200 (1,000 W), largest err / bound, fp16 / bf16 build:
    x 0.030 / 0.030, h 0.988 / 0.995."""
    L = _lib()
    M, K = shape
    g = _gen(M + K + 7 * LN_KINDS.index(kind))
    A = torch.randn(M, K, device='cuda', generator=g).to(_act())
    W = (torch.randn(D, K, device='cuda', generator=g) / math.sqrt(K)).to(_act())
    bias = torch.randn(D, device='cuda', generator=g)
    x_in = _rows(M, D, kind, g)
    lw, lb = _ln_params(D, g)
    xbuf, x = _nan_buf(M, D, torch.float32)
    x.copy_(x_in)
    hbuf, h = _nan_buf(M, D, _act())
    L.check(L.lib.vited_op_gemm_resid_ln(_ptr(A), _ptr(W), _ptr(bias), _ptr(x), _ptr(lw), _ptr(lb), _ptr(h), M, D, K,
                                         LN_EPS, _stream()), 'op_gemm_resid_ln')
    torch.cuda.synchronize()
    _assert_guard(xbuf, M, 'x')
    _assert_guard(hbuf, M, 'h')
    A64, W64, b64 = A.double(), W.double(), bias.double()
    _check_ln_out(f'gemm_resid_ln {M}x{K}', x_in, x, lambda sl: A64[sl] @ W64.t() + b64,
                  lambda sl, xi: (K + 3) * E32 * (A64[sl].abs() @ W64.abs().t() + b64.abs() + xi.abs()), h, lw, lb, PIVOTS)


def _mlp_dx(h_in64, W1, b1, W2, b2):
    """(reference fc2(GELU(fc1(h))) + b2 with the hidden activations rounded to 16 bits, its error bound without the
    x term): the hidden values are rounded where the kernel rounds them; the kernel's pre-rounding value is within
    GELU_ERR + 1.13 (384 + 2) 2^-24 (|h| |W1|^T + |b1|) of the exact one (|GELU'| <= 1.13), so a hidden value next to
    a rounding boundary may round the other way (_flips), and the fc2 accumulation adds (hidden + 3) 2^-24 sum|hid w2|"""
    z = h_in64 @ W1.t() + b1
    gz = torch.nn.functional.gelu(z)
    del z
    eps_g = GELU_ERR + 1.13 * (h_in64.shape[1] + 2) * E32 * (h_in64.abs() @ W1.abs().t() + b1.abs())
    flips = _flips(gz, eps_g)
    hid = _r16(gz)
    del gz, eps_g
    HID = W1.shape[0]
    dx = hid @ W2.t() + b2
    bound = flips @ W2.abs().t() + (HID + 3) * E32 * (hid.abs() @ W2.abs().t() + b2.abs())
    return dx, bound


MLP_SHAPES = [(256, 1536), (70000, 1536), (33333, 1536), (1, 1536), (300, 64), (40000, 192), (262144 + 77, 1536)]


@pytest.mark.parametrize('kind', LN_KINDS)
@pytest.mark.parametrize('shape', MLP_SHAPES, ids=lambda s: 'x'.join(map(str, s)))
def test_mlp_resid_ln_float64(shape, kind):
    """x += fc2(GELU(fc1(h_in))) + b2; h_out = LayerNorm(x), h_out aliasing h_in (mlp_ln.cu). x - prefill: _mlp_dx's
    bound (hidden values that may round the other way + fp32 accumulation) + 3 2^-24 |x|. h: _h_bound, carrying the
    measured error of x. Measured on a B200 (1,000 W), largest err / bound, fp16 / bf16 build: x 0.29 / 0.70,
    h 0.93 / 0.98."""
    L = _lib()
    M, HID = shape
    g = _gen(M + HID + 7 * LN_KINDS.index(kind))
    hbuf, h = _nan_buf(M, D, _act())
    h.copy_(torch.randn(M, D, device='cuda', generator=g).to(_act()))
    h_in64 = h.double()
    W1 = (torch.randn(HID, D, device='cuda', generator=g) / math.sqrt(D)).to(_act())
    b1 = 0.5 * torch.randn(HID, device='cuda', generator=g)
    W2 = (torch.randn(D, HID, device='cuda', generator=g) / math.sqrt(HID)).to(_act())
    b2 = torch.randn(D, device='cuda', generator=g)
    x_in = _rows(M, D, kind, g)
    lw, lb = _ln_params(D, g)
    xbuf, x = _nan_buf(M, D, torch.float32)
    x.copy_(x_in)
    L.check(L.lib.vited_op_mlp_resid_ln(_ptr(h), _ptr(W1), _ptr(b1), _ptr(W2), _ptr(b2), _ptr(x), _ptr(lw), _ptr(lb),
                                        _ptr(h), M, D, HID, LN_EPS, _stream()), 'op_mlp_resid_ln')
    torch.cuda.synchronize()
    _assert_guard(xbuf, M, 'x')
    _assert_guard(hbuf, M, 'h')
    W1d, b1d, W2d, b2d = W1.double(), b1.double(), W2.double(), b2.double()
    cache = {}

    def ref(sl):
        cache[sl.start] = _mlp_dx(h_in64[sl], W1d, b1d, W2d, b2d)
        return cache[sl.start][0]

    _check_ln_out(f'mlp_resid_ln {M}x{HID}', x_in, x, ref,
                  lambda sl, xi: cache.pop(sl.start)[1] + 3 * E32 * xi.abs(), h, lw, lb, PIVOTS)


CPROJ_SHAPES = [(256, 1536), (33333, 1536), (70000, 1536), (262144 + 77, 1536), (1, 1536), (100, 1536), (300, 64),
                (40000, 192)]


@pytest.mark.parametrize('kind', LN_KINDS)
@pytest.mark.parametrize('shape', CPROJ_SHAPES, ids=lambda s: 'x'.join(map(str, s)))
def test_cproj_mlp_resid_ln_float64(shape, kind):
    """x_mid = x + o Wp^T + bp; h2 = round16(norm2(x_mid)); x = x_mid + fc2(GELU(fc1(h2))) + b2; h = norm1'(x)
    (mlp_ln.cu with its prologue). The chain of bounds: x_mid within (384 + 3) 2^-24 (|o| |Wp|^T + |bp| + |x|); h2 is a
    16-bit rounding of a value within _ln_terms of norm2(x_mid_ref), so an element next to a boundary may round the
    other way (_flips); that moves fc1's output by flips |W1|^T, which widens the GELU window of _mlp_dx. x - prefill:
    the sum of these terms; h: _h_bound with the measured error of x.
    Measured on a B200 (1,000 W), largest err / bound, fp16 / bf16 build:
    x 0.013 / 0.053, h 0.93 / 0.99."""
    L = _lib()
    M, HID = shape
    g = _gen(M + HID + 7 * LN_KINDS.index(kind))
    r = lambda *s: torch.randn(*s, device='cuda', generator=g)
    o = r(M, D).to(_act())
    Wp = (r(D, D) / math.sqrt(D)).to(_act())
    bp = r(D)
    W1 = (r(HID, D) / math.sqrt(D)).to(_act())
    b1 = 0.5 * r(HID)
    W2 = (r(D, HID) / math.sqrt(HID)).to(_act())
    b2 = r(D)
    x_in = _rows(M, D, kind, g)
    ln2 = _ln_params(D, g)
    ln1 = _ln_params(D, g)
    xbuf, x = _nan_buf(M, D, torch.float32)
    x.copy_(x_in)
    hbuf, h = _nan_buf(M, D, _act())
    o_in = o.clone()
    L.check(L.lib.vited_op_cproj_mlp_resid_ln(_ptr(o), _ptr(Wp), _ptr(bp), _ptr(x), _ptr(ln2[0]), _ptr(ln2[1]), _ptr(W1),
                                              _ptr(b1), _ptr(W2), _ptr(b2), _ptr(ln1[0]), _ptr(ln1[1]), _ptr(h), M, D,
                                              HID, LN_EPS, _stream()), 'op_cproj_mlp_resid_ln')
    torch.cuda.synchronize()
    assert torch.equal(o, o_in), 'o is an input'
    _assert_guard(xbuf, M, 'x')
    _assert_guard(hbuf, M, 'h')
    o64, Wp64, bp64 = o.double(), Wp.double(), bp.double()
    W1d, b1d, W2d, b2d = W1.double(), b1.double(), W2.double(), b2.double()
    cache = {}

    def ref(sl):
        xi = x_in[sl].double()
        x_mid = xi + o64[sl] @ Wp64.t() + bp64
        e_mid = (D + 3) * E32 * (o64[sl].abs() @ Wp64.abs().t() + bp64.abs() + xi.abs())
        h2_exact, t2 = _ln_terms(x_mid, e_mid, *ln2, PIVOTS)
        h2_flips = _flips(h2_exact, t2)
        h2 = _r16(h2_exact)
        del h2_exact, t2
        z = h2 @ W1d.t() + b1d
        gz = torch.nn.functional.gelu(z)
        del z
        eps_z = (D + 2) * E32 * (h2.abs() @ W1d.abs().t() + b1d.abs()) + h2_flips @ W1d.abs().t()
        hid_flips = _flips(gz, GELU_ERR + 1.13 * eps_z)
        hid = _r16(gz)
        del gz, eps_z
        mlp = hid @ W2d.t() + b2d
        bound = e_mid + hid_flips @ W2d.abs().t() + (HID + 3) * E32 * (hid.abs() @ W2d.abs().t() + b2d.abs() + x_mid.abs())
        cache[sl.start] = bound
        return x_mid - xi + mlp

    _check_ln_out(f'cproj_mlp_resid_ln {M}x{HID}', x_in, x, ref, lambda sl, xi: cache.pop(sl.start), h, *ln1, PIVOTS)


# ---- exactly representable rows -------------------------------------------------------------------------------
def _exact_rows(M, width, pattern, g):
    """rows c + s * sign with s = 2^k (k in [-2, 5]), c = m s (m in [-3, 3]): every value, the mean (c) and the variance
    (s^2) are exact in fp32 in any summation order, and LayerNorm(row) = sign * s / sqrt(s^2 + 1e-6), which is within
    2^-13 of +-1 and so rounds to exactly +-1 in both 16-bit types.
      'within':  signs alternate inside every 32-column group, so every group mean is c (all variance within groups);
      'between': signs constant inside every quarter row (+, +, -, - or a permutation with two of each): the 192-column
                 halves and the 96-column quarters are constant, so the whole variance is the Chan between-group term."""
    k = torch.randint(-2, 6, (M, 1), device='cuda', generator=g).double()
    s = torch.pow(2.0, k)
    c = torch.randint(-3, 4, (M, 1), device='cuda', generator=g).double() * s
    if pattern == 'within':
        sign = torch.ones(width, device='cuda', dtype=torch.float64)
        sign[1::2] = -1
        sign = sign.expand(M, width)
    else:
        perms = torch.tensor([[1, 1, -1, -1], [1, -1, 1, -1], [1, -1, -1, 1], [-1, 1, 1, -1], [-1, 1, -1, 1],
                              [-1, -1, 1, 1]], device='cuda', dtype=torch.float64)
        sign = perms[torch.randint(0, 6, (M,), device='cuda', generator=g)].repeat_interleave(width // 4, dim=1)
    return (c + s * sign).float(), sign


EXACT_KERNELS = ['resid_ln384', 'resid_ln768', 'resid_ln32', 'resid_ln96', 'gemm_resid_ln', 'mlp_resid_ln',
                 'cproj_mlp_resid_ln']


def _run_exact(kernel, x, lw, lb, g):
    """run one LayerNorm kernel on rows x with every other contribution exactly zero (delta = 0, W = Wp = W2 = 0, zero
    biases); returns h (x is updated in place and must come back unchanged)"""
    L = _lib()
    M, width = x.shape
    hbuf, h = _nan_buf(M, width, _act())
    z16 = lambda *s: torch.zeros(*s, dtype=_act(), device='cuda')
    z32 = lambda *s: torch.zeros(*s, device='cuda')
    if kernel.startswith('resid_ln'):
        L.check(L.lib.vited_op_resid_ln(_ptr(x), _ptr(z16(M, width)), _ptr(lw), _ptr(lb), _ptr(h), M, 1, 0, width,
                                        LN_EPS, _stream()), 'op_resid_ln')
    elif kernel == 'gemm_resid_ln':
        A = torch.randn(M, 192, device='cuda', generator=g).to(_act())
        L.check(L.lib.vited_op_gemm_resid_ln(_ptr(A), _ptr(z16(D, 192)), _ptr(z32(D)), _ptr(x), _ptr(lw), _ptr(lb),
                                             _ptr(h), M, D, 192, LN_EPS, _stream()), 'op_gemm_resid_ln')
    elif kernel == 'mlp_resid_ln':
        h.copy_(torch.randn(M, D, device='cuda', generator=g).to(_act()))
        W1 = (torch.randn(1536, D, device='cuda', generator=g) / math.sqrt(D)).to(_act())
        L.check(L.lib.vited_op_mlp_resid_ln(_ptr(h), _ptr(W1), _ptr(z32(1536)), _ptr(z16(D, 1536)), _ptr(z32(D)),
                                            _ptr(x), _ptr(lw), _ptr(lb), _ptr(h), M, D, 1536, LN_EPS, _stream()),
                'op_mlp_resid_ln')
    else:
        o = torch.randn(M, D, device='cuda', generator=g).to(_act())
        W1 = (torch.randn(1536, D, device='cuda', generator=g) / math.sqrt(D)).to(_act())
        ones, zeros = torch.ones(D, device='cuda'), z32(D)
        L.check(L.lib.vited_op_cproj_mlp_resid_ln(_ptr(o), _ptr(z16(D, D)), _ptr(zeros), _ptr(x), _ptr(ones),
                                                  _ptr(zeros), _ptr(W1), _ptr(z32(1536)), _ptr(z16(D, 1536)),
                                                  _ptr(zeros), _ptr(lw), _ptr(lb), _ptr(h), M, D, 1536, LN_EPS,
                                                  _stream()), 'op_cproj_mlp_resid_ln')
    torch.cuda.synchronize()
    _assert_guard(hbuf, M, 'h')
    return h


@pytest.mark.parametrize('affine', ['unit', 'random'])
@pytest.mark.parametrize('pattern', ['within', 'between'])
@pytest.mark.parametrize('kernel', EXACT_KERNELS)
@pytest.mark.parametrize('epi_warps', ['8', '16'])
def test_layernorm_of_exactly_representable_rows(kernel, pattern, affine, epi_warps, monkeypatch):
    """Rows whose LayerNorm is exactly +-1 (_exact_rows). With ln_w = 1, ln_b = 0 the output must be exactly +-1: a
    variance divided by D - 1 gives +-0.9987 (3 fp16 steps, 1 bf16 step below 1) and fails bit-exactly, and in the
    'between' pattern a lost between-group term of the Chan combination gives a zero variance. With random ln_w / ln_b
    the output is round16(+-w + b) up to one 16-bit step (the fp32 product (v - mean) rstd w + b may round to the
    other neighbour). 4,099 rows: every row of every 128-row tile, and a ragged last tile."""
    if epi_warps == '16' and kernel.startswith('resid_ln'):
        pytest.skip('the epilogue forms only exist in the fused tcgen05 kernels')
    _epi_variant(epi_warps, monkeypatch)
    width = int(kernel[8:]) if kernel.startswith('resid_ln') else D
    M = 4099
    g = _gen(EXACT_KERNELS.index(kernel) * 8 + (pattern == 'between') * 2 + (affine == 'random'))
    x, sign = _exact_rows(M, width, pattern, g)
    x_in = x.clone()
    if affine == 'unit':
        lw, lb = torch.ones(width, device='cuda'), torch.zeros(width, device='cuda')
    else:
        lw, lb = _ln_params(width, g)
    h = _run_exact(kernel, x, lw, lb, g)
    assert torch.equal(x, x_in), 'x + 0 must leave every row unchanged'
    if affine == 'unit':
        bad = h.double() != sign
        assert not bad.any(), f'{int(bad.sum())} elements differ from +-1; first {bad.nonzero()[0].tolist()}: ' \
                              f'{float(h[tuple(bad.nonzero()[0].tolist())])}'
    else:
        want = _r16(sign * lw.double() + lb.double())
        err = (h.double() - want).abs()
        _check(err, _step(want.abs()) * 1.0001 + 2 * _tiny16(), f'{kernel} {pattern}: h vs round16(+-w + b)')


# ---------------------------------------------------------------------------------------------------------------
# 2. GEMM (gemm_tc.cu, and the SIMT debugging kernel)
# ---------------------------------------------------------------------------------------------------------------
GEMM_SHAPES = [
    (128, 128, 64), (256, 384, 384), (1000, 1152, 384), (4160, 384, 384), (777, 1536, 384), (640, 384, 1536),
    (65 * 37, 768, 384), (64 * 9, 384, 192), (300, 384, 768), (5, 32, 32), (130, 96, 3072), (1, 8, 8),
    (129, 1152, 384), (20000, 1152, 384),
    (30000, 1536, 384), (26000, 384, 384), (26001, 384, 192), (19999, 768, 384),
]


@pytest.mark.parametrize('impl', [0, 1], ids=['tcgen05', 'simt'])
@pytest.mark.parametrize('act', [0, 1], ids=['none', 'gelu'])
@pytest.mark.parametrize('shape', GEMM_SHAPES, ids=lambda s: 'x'.join(map(str, s)))
def test_gemm_float64(shape, act, impl):
    """C = act(A W^T + b), per element: u |ref| (the 16-bit output) + (K + 2) 2^-24 (sum_k |a_k w_k| + |b|) (fp32
    accumulation and the bias add), times max|GELU'| = 1.13 and + 1e-4 (the GELU epilogue) with GELU. NaN rows past C
    must survive. Measured on a B200 (1,000 W), largest err / bound, fp16 / bf16 build: 0.97 / 0.99."""
    L = _lib()
    M, N, K = shape
    if impl == 1 and M * N * K > 3e9:
        pytest.skip('debug kernel: skip the largest shape')
    g = _gen(M * 7 + N * 3 + K)
    A = torch.randn(M, K, device='cuda', generator=g).to(_act())
    W = (torch.randn(N, K, device='cuda', generator=g) / math.sqrt(K)).to(_act())
    bias = torch.randn(N, device='cuda', generator=g)
    cbuf, C = _nan_buf(M, N, _act())
    L.check(L.lib.vited_op_gemm(_ptr(A), _ptr(W), _ptr(bias), _ptr(C), M, N, K, act, impl, _stream()), 'op_gemm')
    torch.cuda.synchronize()
    _assert_guard(cbuf, M, 'C')
    A64, W64, b64 = A.double(), W.double(), bias.double()
    worst = 0.0
    for r0 in range(0, M, CHUNK):
        sl = slice(r0, min(M, r0 + CHUNK))
        z = A64[sl] @ W64.t() + b64
        acc = (K + 2) * E32 * (A64[sl].abs() @ W64.abs().t() + b64.abs())
        ref = torch.nn.functional.gelu(z) if act else z
        pre = 1.13 * acc + GELU_ERR if act else acc
        bound = _u16() * (ref.abs() + pre) + pre + _tiny16()
        worst = max(worst, _check((C[sl].double() - ref).abs(), bound, f'gemm {shape}'))
    _report(f'gemm {M}x{N}x{K} act={act} impl={impl}', err_over_bound=worst)


# ---------------------------------------------------------------------------------------------------------------
# 3. attention (attention.cu: mma.sync + SIMT; attention_tc.cu: tcgen05 attn_p64 / attn_l64)
# ---------------------------------------------------------------------------------------------------------------
def _rowmap(n_seq, n_patch, has_cls):
    """[n_seq, T] split-layout row of logical token s of sequence b (token 0 = the class token when has_cls)"""
    b = torch.arange(n_seq, device='cuda')[:, None]
    s = torch.arange(n_patch + has_cls, device='cuda')[None, :]
    patch = b * n_patch + s - has_cls
    if has_cls:
        return torch.where(s == 0, n_seq * n_patch + b, patch)
    return patch.expand(n_seq, -1)


def _heads(buf, rows, H, hd):
    """[n, T, H*hd] 16-bit rows -> [n, H, T, hd] float64"""
    t = buf[rows].double()
    return t.view(*rows.shape, H, hd).permute(0, 2, 1, 3)


def _attn_ref(q, k, v, scale):
    """float64 softmax(q k^T scale) v and its error bound, per element:
      u |o|                                   the 16-bit output;
      u S, S = sum_j p_j |v_j|                P rounded to 16 bits before P V (tensor-core kernels);
      2 (EPS_EXP + ds) S                      relative error of every exponential, in numerator and normaliser, where
                                              ds = (hd + 2) 2^-24 scale max_j sum_d |q_d k_jd| is the fp32 error of a score;
      2 (Tk + 8) 2^-24 S                      fp32 accumulation of P V and of the normaliser;
      2^-25 sum_j |v_j| / l (fp16 only)       probabilities below the fp16 normal range (l = sum_j exp(s_j - max) >= 1)."""
    s = (q @ k.transpose(-1, -2)) * scale
    s = s - s.amax(-1, keepdim=True)
    e = torch.exp(s)
    del s
    l = e.sum(-1, keepdim=True)
    p = e / l
    del e
    vabs = v.abs()
    o = p @ v
    S = p @ vabs
    del p
    ds = (q.shape[-1] + 2) * E32 * scale * (q.abs() @ k.abs().transpose(-1, -2)).amax(-1, keepdim=True)
    Tk = k.shape[-2]
    u = _u16()
    bound = u * o.abs() + (u + 2 * (EPS_EXP + ds) + 2 * (Tk + 8) * E32) * S + _tiny16() * vabs.sum(-2, keepdim=True) / l \
        + _tiny16()
    return o, bound


def _tile_edges(n, sizes=(64, 128, 256)):
    """first and last index of every tile of the given sizes over [0, n), and n - 1"""
    out = {n - 1}
    for t in sizes:
        for a in range(0, n, t):
            out.update({a, min(n, a + t) - 1})
    return sorted(out)


A_DOM = 24.0   # q . k = 576 on the chosen pairs: 72 nats (head_dim 64) / 102 nats (head_dim 32) above every other score


def _dominate(q16, k16, qrow, krow, kv_of, triples, H, hd):
    """For every (sequence b, query token sq, head h, key token sk): q of (b, sq, h) becomes A_DOM e_d and, among the
    keys of b's key/value sequence, only key sk keeps a non-zero component d (= A_DOM); d is distinct for every triple
    of one (key/value sequence, head). All other scores of that query row are then exactly 0, so the output row must be
    v of key sk up to one 16-bit rounding. Returns the triples actually placed."""
    used, dirs, placed = set(), {}, []
    for b, sq, h, sk in triples:
        for dh in range(H):
            hh = (h + dh) % H
            if (b, sq, hh) not in used:
                break
        else:
            continue
        c = kv_of(b)
        d = dirs.get((c, hh), 0)
        if d >= hd:
            continue
        dirs[(c, hh)] = d + 1
        used.add((b, sq, hh))
        col = hh * hd
        q16[qrow[b, sq], col:col + hd] = 0
        q16[qrow[b, sq], col + d] = A_DOM
        k16[krow[c], col + d] = 0
        k16[krow[c, sk], col + d] = A_DOM
        placed.append((b, sq, hh, sk))
    return placed


def _dominant_triples(n_seq, H, q_rows, k_keys):
    n = max(len(q_rows), len(k_keys))
    return [(i % n_seq, q_rows[i % len(q_rows)], (i // n_seq) % H, k_keys[(i * 7) % len(k_keys)]) for i in range(n)] + \
        [(i % n_seq, q_rows[(i * 5) % len(q_rows)], (i // n_seq + 1) % H, k_keys[i % len(k_keys)]) for i in range(n)]


def _assert_covered(placed, q_rows, k_keys):
    assert {t[1] for t in placed} == set(q_rows) and {t[3] for t in placed} == set(k_keys), \
        'not every chosen query row and key was placed'


def _check_dominant(o_log, v_log, placed, kvidx, what):
    """o_log [n, H, Tq, hd], v_log [n_kv, H, Tk, hd]: the chosen rows equal the dominant key's v up to one rounding"""
    for b, sq, h, sk in placed:
        got = o_log[b, h, sq]
        want = v_log[kvidx[b], h, sk]
        err = (got - want).abs()
        assert (err <= _u16() * want.abs() + _tiny16()).all(), \
            f'{what}: query (seq {b}, token {sq}, head {h}) does not return key {sk}: max err {float(err.max()):.4g}'


SELF_CFGS = [
    (7, 12, 32, 64, 1), (1, 1, 32, 64, 1), (333, 12, 32, 64, 1), (150, 5, 32, 64, 0), (3, 5, 32, 64, 1),
    (2000, 12, 32, 64, 1), (40, 6, 64, 1024, 1), (1, 1, 64, 256, 1), (9, 3, 64, 512, 0), (30, 2, 64, 256, 1),
    (3, 6, 64, 1024, 1), (5, 12, 32, 64, 0), (2, 6, 64, 1024, 0), (4, 1, 32, 4, 1), (3, 3, 32, 16, 1), (2, 2, 64, 100, 1),
    (1, 2, 32, 130, 0),
]
CROSS_CFGS = [
    (9, 4, 12, 32, 64), (1, 1, 12, 32, 64), (401, 7, 12, 32, 64), (7, 3, 5, 32, 64), (1500, 9, 12, 32, 64),
    (37, 5, 6, 64, 1024), (3, 2, 1, 64, 256), (5, 3, 6, 64, 1024), (6, 2, 1, 32, 4), (4, 4, 2, 64, 16),
]
DOMINANT_SELF = [(3, 6, 64, 1024, 1), (7, 12, 32, 64, 1), (9, 3, 64, 512, 0), (1, 2, 32, 130, 0), (2, 2, 64, 100, 1)]
DOMINANT_CROSS = [(5, 3, 6, 64, 1024), (9, 4, 12, 32, 64), (3, 2, 1, 64, 256)]


def _kv_index(P, n_ctx, g):
    """a permuted, repeated key/value sequence index (every context sequence used when P >= n_ctx)"""
    base = torch.arange(P, device='cuda') % n_ctx
    return base[torch.randperm(P, device='cuda', generator=g)].to(torch.int32)


def _run_self(cfg, impl, dominant, seed):
    L = _lib()
    n_seq, H, hd, n_patch, has_cls = cfg
    Dm = H * hd
    rows = n_seq * n_patch + (n_seq if has_cls else 0)
    g = _gen(seed)
    qkv = torch.randn(rows, 3 * Dm, device='cuda', generator=g).to(_act())
    rm = _rowmap(n_seq, n_patch, has_cls)
    placed = []
    if dominant:
        q_rows = ([0] if has_cls else []) + [t + has_cls for t in _tile_edges(n_patch)]
        k_keys = ([0] if has_cls else []) + [t + has_cls for t in _tile_edges(n_patch, (64, 128))]
        placed = _dominate(qkv[:, :Dm], qkv[:, Dm:2 * Dm], rm, rm, lambda b: b,
                           _dominant_triples(n_seq, H, q_rows, k_keys), H, hd)
        _assert_covered(placed, q_rows, k_keys)
    obuf, o = _nan_buf(rows, Dm, _act())
    st = L.lib.vited_op_attention(_ptr(qkv), 3 * Dm, ctypes.c_void_p(qkv.data_ptr() + 2 * Dm), 3 * Dm,
                                  ctypes.c_void_p(qkv.data_ptr() + 4 * Dm), 3 * Dm, _ptr(o), Dm, n_seq, H, hd, n_patch,
                                  has_cls, n_patch, has_cls, n_seq, None, hd ** -0.5, impl, _stream())
    L.check(st, 'op_attention')
    torch.cuda.synchronize()
    _assert_guard(obuf, rows, 'o')
    q, k, v = (_heads(qkv[:, i * Dm:(i + 1) * Dm], rm, H, hd) for i in range(3))
    return o, rm, (q, k, v), placed, list(range(n_seq))


def _run_cross(cfg, impl, dominant, seed):
    L = _lib()
    P, n_ctx, H, hd, n_patch = cfg
    Dm = H * hd
    rows = P * (n_patch + 1)
    g = _gen(seed)
    qb = torch.randn(rows, Dm, device='cuda', generator=g).to(_act())
    kv = torch.randn(n_ctx * n_patch, 2 * Dm, device='cuda', generator=g).to(_act())
    idx = _kv_index(P, n_ctx, g)
    qm, km = _rowmap(P, n_patch, 1), _rowmap(n_ctx, n_patch, 0)
    idx_l = idx.tolist()
    placed = []
    if dominant:
        q_rows = [0] + [t + 1 for t in _tile_edges(n_patch)]
        k_keys = _tile_edges(n_patch, (64, 128))
        placed = _dominate(qb, kv[:, :Dm], qm, km, lambda b: idx_l[b], _dominant_triples(P, H, q_rows, k_keys), H, hd)
        _assert_covered(placed, q_rows, k_keys)
    obuf, o = _nan_buf(rows, Dm, _act())
    st = L.lib.vited_op_attention(_ptr(qb), Dm, _ptr(kv), 2 * Dm, ctypes.c_void_p(kv.data_ptr() + 2 * Dm), 2 * Dm,
                                  _ptr(o), Dm, P, H, hd, n_patch, 1, n_patch, 0, n_ctx, _ptr(idx), hd ** -0.5, impl,
                                  _stream())
    L.check(st, 'op_attention')
    torch.cuda.synchronize()
    _assert_guard(obuf, rows, 'o')
    q = _heads(qb, qm, H, hd)
    k = _heads(kv[:, :Dm], km, H, hd)[idx.long()]
    v = _heads(kv[:, Dm:], km, H, hd)[idx.long()]
    return o, qm, (q, k, v), placed, idx_l


def _check_attention(name, o, qm, qkv, placed, H, hd, scale, seq_block=64):
    """o (16-bit, split layout) against _attn_ref, sequence block by sequence block; then the dominant rows"""
    q, k, v = qkv
    worst = 0.0
    for b0 in range(0, q.shape[0], seq_block):
        sb = slice(b0, b0 + seq_block)
        ref, bound = _attn_ref(q[sb], k[sb], v[sb], scale)
        got = _heads(o, qm[sb], H, hd)
        assert torch.isfinite(got).all(), f'{name}: non-finite output'
        worst = max(worst, _check((got - ref).abs(), bound, f'{name}, sequences {b0}+'))
    if placed:
        o_log = _heads(o, qm, H, hd)
        _check_dominant(o_log, v, placed, list(range(q.shape[0])), name)
    _report(name, err_over_bound=worst)
    return worst


IMPLS = [0, 1, 2]
IMPL_IDS = ['fast', 'simt', 'mma_sync']


@pytest.mark.parametrize('impl', IMPLS, ids=IMPL_IDS)
@pytest.mark.parametrize('cfg', SELF_CFGS, ids=lambda c: 'x'.join(map(str, c)))
def test_self_attention_float64(cfg, impl):
    """Self-attention (q / k / v column slices of one qkv buffer, split layout) against _attn_ref's per-element bound.
    At 1,025 tokens |o| is ~0.05 (0.64 at most) and S ~0.8: the bound, ~(u + 3e-4) S, fails on a 1 % scale error of o.
    Measured on a B200 (1,000 W), largest err / bound, fp16 / bf16 build: 0.49 / 0.60."""
    n_seq, H, hd, n_patch, has_cls = cfg
    o, qm, qkv, placed, _ = _run_self(cfg, impl, False, sum(cfg))
    _check_attention(f'self {cfg} impl={impl}', o, qm, qkv, placed, H, hd, hd ** -0.5, 8 if hd == 64 else 256)


@pytest.mark.parametrize('impl', IMPLS, ids=IMPL_IDS)
@pytest.mark.parametrize('cfg', CROSS_CFGS, ids=lambda c: 'x'.join(map(str, c)))
def test_cross_attention_float64(cfg, impl):
    """Cross-attention (queries with a class token, patch-only keys picked through a permuted, repeated kv_index)
    against _attn_ref's per-element bound. Measured on a B200 (1,000 W), largest err / bound, fp16 / bf16 build: 0.48 /
    0.57."""
    P, n_ctx, H, hd, n_patch = cfg
    o, qm, qkv, placed, idx = _run_cross(cfg, impl, False, sum(cfg))
    _check_attention(f'cross {cfg} impl={impl}', o, qm, qkv, placed, H, hd, hd ** -0.5, 8 if hd == 64 else 256)


@pytest.mark.parametrize('impl', IMPLS, ids=IMPL_IDS)
@pytest.mark.parametrize('cfg', DOMINANT_SELF, ids=lambda c: 'x'.join(map(str, c)))
def test_self_attention_dominant_keys(cfg, impl):
    """One key dominates chosen query rows by >= 72 nats (_dominate): the query rows are the class token and the first
    and last row of every 64-, 128- and 256-row tile; the keys are the class-token key and the first and last key of
    every 64- and 128-key tile. Each chosen row must return exactly its key's v row (an off-by-one row, a wrong head
    column or a misplaced class token shows at once); the jump of the running maximum also drives the lazy rescale of
    the tcgen05 kernel. The whole output is also held to _attn_ref's bound.
    Measured on a B200 (1,000 W), largest err / bound, fp16 / bf16 build:
    0.56 / 0.75."""
    n_seq, H, hd, n_patch, has_cls = cfg
    o, qm, qkv, placed, _ = _run_self(cfg, impl, True, 100 + sum(cfg))
    _check_attention(f'self dominant {cfg} impl={impl}', o, qm, qkv, placed, H, hd, hd ** -0.5, 8)


@pytest.mark.parametrize('impl', IMPLS, ids=IMPL_IDS)
@pytest.mark.parametrize('cfg', DOMINANT_CROSS, ids=lambda c: 'x'.join(map(str, c)))
def test_cross_attention_dominant_keys(cfg, impl):
    """test_self_attention_dominant_keys for cross-attention with a permuted, repeated kv_index: a wrong kv_index entry
    returns another context sequence's v row.
    Measured on a B200 (1,000 W), largest err / bound, fp16 / bf16 build: 0.59 / 0.75."""
    P, n_ctx, H, hd, n_patch = cfg
    o, qm, qkv, placed, idx = _run_cross(cfg, impl, True, 200 + sum(cfg))
    _check_attention(f'cross dominant {cfg} impl={impl}', o, qm, qkv, placed, H, hd, hd ** -0.5, 8)


# ---------------------------------------------------------------------------------------------------------------
# 4. class-token-only attention (attention_cls: attn_cls_warp_kernel, attn_p64_kernel in cls mode, attn_mma_kernel
#    with cls_only = 1)
# ---------------------------------------------------------------------------------------------------------------
# (name, n_seq, n_kv_seq (None: self-attention with the class-token key), H, hd, n_patch)
CLS_CASES = {
    'puzzle_self': (333, None, 12, 32, 64),
    'puzzle_cross': (401, 7, 12, 32, 64),
    'hisfrag_self': (8, None, 6, 64, 1024),
    'hisfrag_cross': (7, 3, 6, 64, 1024),
}


def _check_attention_cls(case):
    """q [rows, D] and k | v [rows_kv, 2D] as the pruned tail of decode_chunk lays them out (engine.cu); the class-token
    query of every sequence is made to pick a dominant key in some head (the class-token key included)."""
    L = _lib()
    n_seq, n_kv, H, hd, n_patch = CLS_CASES[case]
    self_attn = n_kv is None
    k_cls = 1 if self_attn else 0
    n_kv = n_seq if self_attn else n_kv
    Dm = H * hd
    rows = n_seq * (n_patch + 1)
    kv_rows = n_kv * (n_patch + k_cls)
    g = _gen(len(case) * 31 + n_seq)
    q = torch.randn(rows, Dm, device='cuda', generator=g).to(_act())
    kv = torch.randn(kv_rows, 2 * Dm, device='cuda', generator=g).to(_act())
    idx = None if self_attn else _kv_index(n_seq, n_kv, g)
    idx_l = list(range(n_seq)) if self_attn else idx.tolist()
    qm, km = _rowmap(n_seq, n_patch, 1), _rowmap(n_kv, n_patch, k_cls)
    keys = ([0] if k_cls else []) + [t + k_cls for t in _tile_edges(n_patch, (64, 128))]
    triples = [(i % n_seq, 0, (i // n_seq) % H, sk) for i, sk in enumerate(keys)]
    placed = _dominate(q, kv[:, :Dm], qm, km, lambda b: idx_l[b], triples, H, hd)
    assert {sk for _, _, _, sk in placed} == set(keys), 'not every chosen key was placed'
    scale = hd ** -0.5
    obuf, o = _nan_buf(rows, Dm, _act())
    L.check(L.lib.vited_op_attention_cls(_ptr(q), Dm, _ptr(kv), 2 * Dm, ctypes.c_void_p(kv.data_ptr() + 2 * Dm), 2 * Dm,
                                         _ptr(o), Dm, n_seq, H, hd, n_patch, k_cls, n_kv, _ptr(idx), scale, _stream()),
            'op_attention_cls')
    torch.cuda.synchronize()
    cls0 = n_seq * n_patch
    assert torch.isnan(o[:cls0].float()).all(), 'a patch row of o was written'
    _assert_guard(obuf, rows, 'o')
    # float64 reference of the class-token query rows only
    qc = _heads(q, qm[:, :1], H, hd)
    k = _heads(kv[:, :Dm], km, H, hd)[idx_l]
    v = _heads(kv[:, Dm:], km, H, hd)[idx_l]
    worst = 0.0
    for b0 in range(0, n_seq, 64):
        sb = slice(b0, b0 + 64)
        ref, bound = _attn_ref(qc[sb], k[sb], v[sb], scale)
        got = _heads(o, qm[sb, :1], H, hd)
        worst = max(worst, _check((got - ref).abs(), bound, f'attention_cls {case}, sequences {b0}+'))
    _check_dominant(_heads(o, qm[:, :1], H, hd), v, placed, list(range(n_seq)), f'attention_cls {case}')
    # the same rows from the full attention kernel on the same inputs: both within their bound of the reference
    fbuf, full = _nan_buf(rows, Dm, _act())
    L.check(L.lib.vited_op_attention(_ptr(q), Dm, _ptr(kv), 2 * Dm, ctypes.c_void_p(kv.data_ptr() + 2 * Dm), 2 * Dm,
                                     _ptr(full), Dm, n_seq, H, hd, n_patch, 1, n_patch, k_cls, n_kv, _ptr(idx), scale,
                                     0, _stream()), 'op_attention')
    torch.cuda.synchronize()
    for b0 in range(0, n_seq, 64):
        sb = slice(b0, b0 + 64)
        _, bound = _attn_ref(qc[sb], k[sb], v[sb], scale)
        diff = (_heads(o, qm[sb, :1], H, hd) - _heads(full, qm[sb, :1], H, hd)).abs()
        _check(diff, 2 * bound, f'attention_cls {case} vs vited_op_attention, sequences {b0}+')
    _report(f'attention_cls {case} (VITED_ATTN_CLS_WARP={os.environ.get("VITED_ATTN_CLS_WARP", "")}, '
            f'VITED_ATTN_TC={os.environ.get("VITED_ATTN_TC", "")})', err_over_bound=worst)


CLS_KERNELS = {
    # kernel -> environment (both variables are read once per process: the non-default kernels run in a subprocess)
    'warp': {},
    'tcgen05': {'VITED_ATTN_CLS_WARP': '0'},
    'mma_sync': {'VITED_ATTN_CLS_WARP': '0', 'VITED_ATTN_TC': '0'},
}


@pytest.mark.parametrize('kernel', list(CLS_KERNELS))
@pytest.mark.parametrize('case', ['puzzle_self', 'puzzle_cross'])
def test_attention_cls_puzzle_shape(case, kernel):
    """The class-token query rows of the pruned last layer at the puzzle shape (64 + 1 tokens, head_dim 32), through
    each of its three kernels: attn_cls_warp_kernel (default), attn_p64_kernel in cls mode, attn_mma_kernel with
    cls_only = 1. Checks: _attn_ref's bound; every patch row of o keeps its NaN; a dominant key (the class-token key,
    keys 0 / 63 / last) comes back exactly; the rows agree with vited_op_attention within twice the bound.
    Measured on a B200 (1,000 W), largest err / bound, fp16 / bf16 build: 0.43 / 0.45."""
    env = CLS_KERNELS[kernel]
    if not env:
        _check_attention_cls(case)
        return
    from tests.conftest import ROOT
    code = ("import sys; sys.path.insert(0, %r)\n"
            "from tests.test_gpu_score_kernels import _check_attention_cls\n"
            "_check_attention_cls(%r)\n") % (ROOT, case)
    r = subprocess.run([sys.executable, '-c', code], env=dict(os.environ, **env), capture_output=True, text=True,
                       timeout=600)
    print(r.stdout[-2000:])
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]


@pytest.mark.parametrize('case', ['hisfrag_self', 'hisfrag_cross'])
def test_attention_cls_hisfrag_shape(case):
    """The Hisfrag20 shape (1,024 + 1 tokens, head_dim 64): attn_mma_kernel with cls_only = 1, the kernel the model's
    pruned last layer runs. Checks as test_attention_cls_puzzle_shape, with dominant keys at the class token and the
    first and last key of every 64- and 128-key tile.
    Measured on a B200 (1,000 W), largest err / bound, fp16 / bf16 build: 0.10 / 0.13."""
    _check_attention_cls(case)


# ---------------------------------------------------------------------------------------------------------------
# 5. final LayerNorm + head (head_kernel, rowops.cu)
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('with_delta', [False, True], ids=['x', 'x+delta'])
@pytest.mark.parametrize('C', [1, 4])
@pytest.mark.parametrize('width', [384, 32])
@pytest.mark.parametrize('P', [1, 3001])
def test_head_float64(P, width, C, with_delta):
    """logits = LayerNorm(x + delta) w + b, then . head_w + head_b, all in fp32 (one warp per row). Rows carry a
    common offset of 50 on a unit spread. Bound per logit:
      * the statistics (sums along chains of at most D/32 + 5 additions, n = D/32 + 8): the mean error is common to the
        row, so it moves the logit by |d mean| rstd |sum_d w_d hw_d|, |d mean| <= n 2^-24 mean|v|; the relative rstd
        error (n 2^-24 + 2^-21, two-pass variance) moves it by that times |sum_d xhat_d w_d hw_d|;
      * the per-element y = (v - mean) rstd w + b (4 2^-24 |y|) and the dot product ((n + 1) 2^-24 sum |y hw|);
      * the addition of delta to x: 2^-24 |x + delta| rstd |w hw|.
    No 16-bit rounding anywhere, so a variance divided by D - 1 (a 1.3e-3 relative shift at D = 384) fails in every
    build. NaN past the P * C logits must survive.
    Measured on a B200 (1,000 W), largest err / bound, fp16 / bf16 build: 0.21 / 0.22."""
    L = _lib()
    g = _gen(P + width + C + with_delta)
    x = torch.randn(P, width, device='cuda', generator=g) + 50 * (1 + torch.rand(P, 1, device='cuda', generator=g))
    delta = torch.randn(P, width, device='cuda', generator=g).to(_act()) if with_delta else None
    lw, lb = _ln_params(width, g)
    hw = torch.randn(C, width, device='cuda', generator=g) / math.sqrt(width)
    hb = torch.randn(C, device='cuda', generator=g)
    out = torch.full((P * C + GUARD,), float('nan'), device='cuda')
    L.check(L.lib.vited_op_head(_ptr(x), _ptr(delta), _ptr(lw), _ptr(lb), _ptr(hw), _ptr(hb), _ptr(out), P, width, C,
                                LN_EPS, _stream()), 'op_head')
    torch.cuda.synchronize()
    assert torch.isnan(out[P * C:]).all(), 'the head wrote past its P * C logits'
    v = x.double() + (delta.double() if with_delta else 0)
    w64, b64, hw64 = lw.double(), lb.double(), hw.double()
    y, xhat, rstd = _ln64(v, w64, b64)
    ref = y @ hw64.t() + hb.double()
    n = width // 32 + 8
    dmean = n * E32 * v.abs().mean(1, keepdim=True)
    drel = n * E32 + RSQRT_ERR
    bound = dmean * rstd * (w64 @ hw64.t()).abs() + drel * ((xhat * w64) @ hw64.t()).abs() \
        + (4 + n + 1) * E32 * (y.abs() @ hw64.abs().t()) + E32 * ref.abs() \
        + (E32 * v.abs() * rstd) @ (w64[:, None] * hw64.t()).abs()
    worst = _check((out[:P * C].view(P, C).double() - ref).abs(), bound, f'head P={P} D={width} C={C}')
    _report(f'head P={P} D={width} C={C} delta={with_delta}', err_over_bound=worst)
