"""GPU: the training iteration after the backward pass (csrc/train_optim.cu, train.train_iteration) -- the range check
that detects saturated 16-bit gradients, the flag-reporting attention backward, the bit-reproducible gradient norm, the
fused AdamW step against torch.optim.AdamW, and the whole iteration against train_step + clip_grad_norm_ + torch AdamW,
including overflow handling, a short learning run against a float64 loop and the scoring engine's weight refresh."""
import ctypes
import math
import os

import numpy as np
import pytest
import torch

from tests import helpers

pytestmark = pytest.mark.gpu

E32 = 2.0 ** -24


def _lib():
    from vited_b200 import _lib
    return _lib


def _act():
    return _lib().act_dtype()


def _fp16():
    return _act() == torch.float16


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


# ---------------------------------------------------------------------------------------------------------------
# range check
# ---------------------------------------------------------------------------------------------------------------
def _range_check(x, n=None, flag_init=0, limit=None):
    lib = _lib()
    flag = torch.full((1,), flag_init, dtype=torch.int32, device='cuda')
    n = x.numel() if n is None else n
    lim = lib.range_limit() if limit is None else limit
    lib.check(lib.lib.vited_train_range_check(_ptr(x), 1 if x.dtype == torch.float32 else 0, n, lim, _ptr(flag), _stream()),
              'range_check')
    return int(flag.item())


def _edge_values(dtype):
    """(values that must pass, values that must be flagged) in this build, for a buffer of ``dtype``"""
    inf = float('inf')
    if _fp16():
        below = 65472.0 if dtype != torch.float32 else float(np.nextafter(np.float32(65504), np.float32(0)))
        return [below, -below, 0.0, 1e-8], [65504.0, -65504.0, inf, -inf, float('nan')]
    big = float(torch.finfo(dtype).max)
    return [big, -big, 0.0], [inf, -inf, float('nan')]


@pytest.mark.parametrize('dtype', ['f32', 'act'])
def test_range_check_edges_and_positions(dtype):
    """Every value just inside the limit passes, every value at it or beyond (and every NaN) sets the flag, wherever
    it sits: scalar head (before the first 16-byte boundary), vector body, scalar tail, at odd element offsets."""
    dt = torch.float32 if dtype == 'f32' else _act()
    ok, bad = _edge_values(dt)
    for off in (0, 1, 3, 5):
        for n in (1, 2, 7, 8, 9, 33, 1000, 4099):
            buf = torch.zeros(off + n + 16, dtype=dt, device='cuda')
            x = buf[off:off + n]
            for v in ok:
                x.fill_(v)
                assert _range_check(x) == 0, (off, n, v)
            x.zero_()
            positions = sorted({0, min(3, n - 1), n // 2, n - 1})
            for pos in positions:
                for v in bad:
                    x[pos] = v
                    assert _range_check(x) == 1, (off, n, pos, v)
                    x[pos] = 0
            buf[off + n:] = float('nan')          # past the end: never read
            assert _range_check(x) == 0, (off, n)


def test_range_check_sizes_and_stickiness():
    dt = _act()
    assert _range_check(torch.empty(0, device='cuda'), n=0) == 0
    assert _range_check(torch.full((4,), float('nan'), device='cuda'), n=0) == 0      # n = 0 reads nothing
    for dtype in (torch.float32, dt):
        x = torch.randn(1_234_567 + 3, device='cuda').to(dtype)[3:]
        assert _range_check(x) == 0
        assert _range_check(x, flag_init=7) == 7        # clean input never writes the flag
        assert _range_check(x, flag_init=1) == 1        # ... so a set flag stays set
        for pos in (0, 1, 611_111, 1_234_566):
            y = x.clone()
            y[pos] = float('inf')
            assert _range_check(y) == 1, pos
            assert _range_check(y[:1] if pos == 0 else y[pos:pos + 1]) == 1
        one = torch.tensor([float('nan')], device='cuda').to(dtype)
        assert _range_check(one) == 1


def test_range_limit_of_the_build():
    assert _lib().range_limit() == (65504.0 if _fp16() else float('inf'))


# ---------------------------------------------------------------------------------------------------------------
# attention backward with the flag
# ---------------------------------------------------------------------------------------------------------------
ATTN_SHAPES = {   # n_seq, heads, hd, Tq, Tk: Hisfrag20 decoder self-attention and cross-attention (2 pairs)
    'hisfrag_self': (2, 6, 64, 1025, 1025),
    'hisfrag_cross': (2, 6, 64, 1025, 1024),
    'hd32': (3, 3, 32, 65, 65),
}


def _attn(n_seq, H, hd, Tq, Tk, q, k, v, d_o, chk, flag=None):
    lib = _lib()
    act = _act()
    o = torch.empty(n_seq * Tq, H * hd, dtype=act, device='cuda')
    lse = torch.empty(n_seq, H, Tq, device='cuda')
    scale = hd ** -0.5
    s = _stream()
    lib.check(lib.lib.vited_train_attention(0, _ptr(q), H * hd, _ptr(k), H * hd, _ptr(v), H * hd, _ptr(o), H * hd, _ptr(lse),
                                            None, 0, None, None, 0, None, 0, None, 0, n_seq, H, hd, Tq, Tk, scale, s), 'fwd')
    dsum = torch.empty(n_seq, H, Tq, device='cuda')
    dq = torch.zeros(n_seq * Tq, H * hd, device='cuda')
    dk = torch.zeros(n_seq * Tk, H * hd, device='cuda')
    dv = torch.zeros(n_seq * Tk, H * hd, device='cuda')
    args = (1, _ptr(q), H * hd, _ptr(k), H * hd, _ptr(v), H * hd, _ptr(o), H * hd, _ptr(lse), _ptr(d_o), H * hd, _ptr(dsum),
            _ptr(dq), H * hd, _ptr(dk), H * hd, _ptr(dv), H * hd, n_seq, H, hd, Tq, Tk, scale)
    if chk:
        lib.check(lib.lib.vited_train_attention_chk(*args, _ptr(flag), s), 'bwd chk')
    else:
        lib.check(lib.lib.vited_train_attention(*args, s), 'bwd')
    return dq, dk, dv, dsum


@pytest.mark.parametrize('case', sorted(ATTN_SHAPES))
def test_attention_chk_is_the_unchecked_backward(case):
    """With a null flag, and with a flag on clean input, the _chk form writes bit-identical dq / dk / dv / dsum; the
    flag stays 0."""
    n_seq, H, hd, Tq, Tk = ATTN_SHAPES[case]
    g = torch.Generator(device='cuda').manual_seed(3)
    q = torch.randn(n_seq * Tq, H * hd, device='cuda', generator=g).to(_act())
    k = torch.randn(n_seq * Tk, H * hd, device='cuda', generator=g).to(_act())
    v = torch.randn(n_seq * Tk, H * hd, device='cuda', generator=g).to(_act())
    d_o = torch.randn(n_seq * Tq, H * hd, device='cuda', generator=g)
    want = _attn(n_seq, H, hd, Tq, Tk, q, k, v, d_o, False)
    null = _attn(n_seq, H, hd, Tq, Tk, q, k, v, d_o, True, None)
    flag = torch.zeros(1, dtype=torch.int32, device='cuda')
    flagged = _attn(n_seq, H, hd, Tq, Tk, q, k, v, d_o, True, flag)
    for a, b, c in zip(want, null, flagged):
        assert torch.equal(a, b) and torch.equal(a, c)
    assert int(flag.item()) == 0


def test_attention_chk_flags_a_saturating_ds():
    """d_o = 16 and V = +-60000 (both in range) with a uniform softmax over 64 keys: dP_j = +-16 * 60000 * 64 and
    |dS| = (1/64) |dP_j - D| / 8 ~ 1.2e5 > 65504 in the fp16 build. A bf16 build represents that value, so there the
    input is clean and the flag must stay 0."""
    n_seq, H, hd, T = 1, 1, 64, 64
    q = torch.zeros(T, hd, dtype=_act(), device='cuda')
    k = torch.zeros(T, hd, dtype=_act(), device='cuda')
    sign = torch.where(torch.arange(T, device='cuda') % 2 == 0, 1.0, -1.0).view(T, 1)
    v = (sign * 60000.0 * torch.ones(T, hd, device='cuda')).to(_act())
    d_o = torch.full((T, hd), 16.0, device='cuda')
    flag = torch.zeros(1, dtype=torch.int32, device='cuda')
    _attn(n_seq, H, hd, T, T, q, k, v, d_o, True, flag)
    assert int(flag.item()) == (1 if _fp16() else 0)
    # the same input through the unchecked entry point: saturated, finite, silently wrong
    dq, dk, dv, _ = _attn(n_seq, H, hd, T, T, q, k, v, d_o, False)
    assert torch.isfinite(dq).all() and torch.isfinite(dk).all()


# ---------------------------------------------------------------------------------------------------------------
# gradient norm
# ---------------------------------------------------------------------------------------------------------------
def _norm_table(tensors):
    return torch.tensor([[t.data_ptr(), t.numel()] for t in tensors], dtype=torch.int64).cuda()


def _grad_norm(tensors, n_partials=148 * 8):
    lib = _lib()
    table = _norm_table(tensors)
    partials = torch.empty(n_partials, dtype=torch.float64, device='cuda')
    out = torch.zeros(2, dtype=torch.int32, device='cuda')
    lib.check(lib.lib.vited_train_grad_norm(_ptr(table), len(tensors), _ptr(partials), n_partials, _ptr(out), _stream()),
              'grad_norm')
    host = out.cpu()
    return float(host[:1].view(torch.float32)), int(host[1])


@pytest.fixture(scope='module')
def hisfrag20_grads():
    _, kw = helpers.load_model_case('hisfrag20_patch16_512')
    shapes = helpers.shapes_from_kwargs(kw)
    g = torch.Generator(device='cuda').manual_seed(1)
    return {k: torch.randn(s, device='cuda', generator=g) * 1e-3 for k, s in shapes.items()}


def test_grad_norm_over_the_hisfrag20_parameter_set(hisfrag20_grads):
    """50.4 M fp32 gradient elements in 300+ tensors down to the 1-element head bias: fp64 partial sums, so the only
    error against float64 is the final rounding to float32 (2^-24 relative); bound 1e-6. Two calls agree bit for bit."""
    ts = list(hisfrag20_grads.values())
    assert sum(t.numel() for t in ts) > 50_000_000 and hisfrag20_grads['head.bias'].numel() == 1
    want = sum(float(t.double().pow(2).sum()) for t in ts)
    got, flag = _grad_norm(ts)
    assert flag == 0
    assert abs(got - want) <= 1e-6 * want, (got, want)
    again, _ = _grad_norm(ts)
    assert again == got
    # a gradient of one element, on its own and at the end of the table
    hb = hisfrag20_grads['head.bias']
    assert _grad_norm([hb])[0] == np.float32(float(hb.double().pow(2).sum()))


def test_grad_norm_reports_inf_and_nan(hisfrag20_grads):
    names = list(hisfrag20_grads)
    for name in (names[0], names[len(names) // 2], 'head.bias'):
        for bad in (float('inf'), float('-inf'), float('nan')):
            t = hisfrag20_grads[name]
            old = t.view(-1)[t.numel() - 1].item()
            t.view(-1)[t.numel() - 1] = bad
            try:
                got, flag = _grad_norm(list(hisfrag20_grads.values()))
            finally:
                t.view(-1)[t.numel() - 1] = old
            assert flag == 1 and not math.isfinite(got), (name, bad)


def test_grad_norm_flags_an_overflowing_sum():
    big = torch.full((4,), 2e19, device='cuda')            # squares sum to 1.6e39: finite in fp64, not in float32
    got, flag = _grad_norm([big])
    assert flag == 1 and got == float('inf')


# ---------------------------------------------------------------------------------------------------------------
# AdamW
# ---------------------------------------------------------------------------------------------------------------
ADAM_SHAPES = [(384, 1536), (1,), (385,), (7, 33), (1025, 384), (3,)]


def _views(buf_len, offsets, shapes, g, fill):
    buf = fill(buf_len, g)
    return buf, [buf[o:o + int(np.prod(s))].view(s) for o, s in zip(offsets, shapes)]


@pytest.mark.parametrize('step', [1, 1000])
def test_adamw_matches_torch(step):
    """One fused step against torch.optim.AdamW(foreach=False, fused=False) on the same fp32 tensors -- views at odd
    element offsets into one buffer per role, a weight-decay group and a wd = 0 group, clip_coef 0.37, step 1 (moments
    zero) and step 1000 (random moments).

    Tolerance: both sides round each of the same ~12 fp32 operations once; they may differ by fused multiply-adds and by
    torch's division by the scalar sqrt(bc2) as a multiplication by its reciprocal. That is a few units of 2^-24
    relative in m, v and the update u = step_size * m / denom; p = p * decay + u then differs by at most a few ulp of
    |p| plus a few ulp of |u|. Bound: 8 * 2^-24 * (|p| + |u|) per element (m, v: 8 * 2^-24 of their magnitude).
    Measured on a B200 (fp16 build): the worst parameter difference is 0.46 of the bound at step 1, 0.26 at step 1000."""
    from vited_b200 import _lib as lib
    g = torch.Generator(device='cuda').manual_seed(step)
    sizes = [int(np.prod(s)) for s in ADAM_SHAPES]
    offsets, o = [], 1
    for n in sizes:
        offsets.append(o)
        o += n + 3                                          # odd offsets, no alignment
    randn = lambda n, g: torch.randn(n, device='cuda', generator=g)
    _, ps = _views(o, offsets, ADAM_SHAPES, g, randn)
    _, gs = _views(o, offsets, ADAM_SHAPES, g, lambda n, g: torch.randn(n, device='cuda', generator=g) * 1e-2)
    _, ms = _views(o, offsets, ADAM_SHAPES, g, lambda n, g: torch.randn(n, device='cuda', generator=g) * 1e-3)
    _, vs = _views(o, offsets, ADAM_SHAPES, g, lambda n, g: torch.rand(n, device='cuda', generator=g) * 1e-5)
    if step == 1:
        for t in ms + vs:
            t.zero_()
    lr, betas, eps, wd, clip = 1e-3, (0.9, 0.999), 1e-8, 0.05, 0.37
    decays = [wd if i % 2 == 0 else 0.0 for i in range(len(ps))]
    # torch on copies
    rp = [torch.nn.Parameter(p.clone()) for p in ps]
    for p, gr in zip(rp, gs):
        p.grad = gr.clone()
        p.grad.mul_(torch.tensor(clip, dtype=torch.float32, device='cuda'))
    ref = torch.optim.AdamW([{'params': [p], 'weight_decay': d} for p, d in zip(rp, decays)], lr=lr, betas=betas, eps=eps,
                            foreach=False, fused=False)
    for p, m, v in zip(rp, ms, vs):
        ref.state[p] = {'step': torch.tensor(float(step - 1)), 'exp_avg': m.clone(), 'exp_avg_sq': v.clone()}
    ref.step()
    grads_before = [t.clone() for t in gs]
    table = torch.tensor([[p.data_ptr(), gr.data_ptr(), m.data_ptr(), v.data_ptr(), p.numel(),
                           int(np.float64(d).view(np.int64))] for p, gr, m, v, d in zip(ps, gs, ms, vs, decays)],
                         dtype=torch.int64).cuda()
    lib.check(lib.lib.vited_train_adamw(_ptr(table), len(ps), max(sizes), lr, betas[0], betas[1], eps, clip,
                                        1 - betas[0] ** step, 1 - betas[1] ** step, _stream()), 'adamw')
    torch.cuda.synchronize()
    worst = 0.0
    bc1, bc2 = 1 - betas[0] ** step, 1 - betas[1] ** step
    for p, m, v, r, gr, gb in zip(ps, ms, vs, rp, gs, grads_before):
        st = ref.state[r]
        u = (lr / bc1) * st['exp_avg'].abs() / (st['exp_avg_sq'].sqrt() / math.sqrt(bc2) + eps)
        bound = 8 * E32 * (r.detach().abs() + u)
        worst = max(worst, float(((p - r.detach()).abs() / bound).max()))
        assert ((p - r.detach()).abs() <= bound).all()
        assert ((m - st['exp_avg']).abs() <= 8 * E32 * st['exp_avg'].abs()).all()
        assert ((v - st['exp_avg_sq']).abs() <= 8 * E32 * st['exp_avg_sq'].abs()).all()
        assert torch.equal(gr, gb)                          # the gradient is read, not written
    print(f'adamw step {step}: worst |p - torch| / bound = {worst:.3g}')


# ---------------------------------------------------------------------------------------------------------------
# the whole iteration
# ---------------------------------------------------------------------------------------------------------------
def _case(name):
    _, kw = helpers.load_model_case(name)
    if name == 'hisfrag20_patch16_512':
        kw = dict(kw, depth=1, c_depth=1)
    return kw


def _models(kw, seed):
    a, sd = helpers.make_gpu_model(kw, seed)
    b, _ = helpers.make_gpu_model(kw, seed)
    return a, b, sd


def _batch(kw, n, seed):
    from vited_b200 import synthetic
    return synthetic.synthetic_images(n, kw['img_size'], seed=seed).cuda()


@pytest.mark.parametrize('name', ['test_patch32_64', 'small_hd64', 'hisfrag20_patch16_512'])
def test_iteration_composes_train_step_clip_and_torch_adamw(name):
    """Two iterations of train_iteration against clip_grad_norm_ + torch AdamW applied to the gradient train_iteration
    itself left in p.grad (the backward pass scatter-adds with atomics, so it is not bit-reproducible and the same
    p.grad is fed to both). The norm agrees to fp32 rounding (fp64 sum vs torch's fp32 norm of norms: 1e-5 relative);
    the parameters to 8 ulp plus 1e-4 lr: Adam's update is lr * m / (sqrt(v) + eps), insensitive to the few-ulp clip
    coefficient difference except where |g| ~ eps. Measured on a B200 (fp16 build): the worst parameter difference is
    0.2 of its bound, the norm within 1e-5 relative."""
    from vited_b200 import train
    kw = _case(name)
    model, ref, _ = _models(kw, 21)
    targets = [0, 0, 0, 1, 1, 1]
    lr = 1e-3
    opt = train.AdamW(model, lr=lr)
    scaler = train.LossScaler(init_scale=1024.0)
    rparams = dict(ref.named_parameters())
    torch_opt = torch.optim.AdamW(opt._torch_groups(rparams), lr=lr, foreach=False, fused=False)
    for it in range(2):
        samples = _batch(kw, len(targets), 50 + it)
        gen = torch.Generator().manual_seed(it)
        out = train.train_iteration(model, samples, targets, opt, scaler, generator=gen)
        loss, logits, groups, labels, norm, skipped = out
        assert not skipped and opt.t == it + 1
        for n, p in model.named_parameters():
            rparams[n].grad = p.grad.clone()
        want = torch.nn.utils.clip_grad_norm_(list(rparams.values()), 5.0)
        assert abs(norm - float(want)) <= 1e-5 * float(want), (norm, float(want))
        torch_opt.step()
        worst = 0.0
        for n, p in model.named_parameters():
            diff = (p.detach() - rparams[n].detach()).abs()
            bound = 8 * E32 * rparams[n].detach().abs() + 1e-4 * lr
            worst = max(worst, float((diff / bound).max()))
            assert (diff <= bound).all(), (it, n, float(diff.max()))
        print(f'{name} iteration {it}: loss {loss.item():.5f}, grad norm {norm:.5g}, worst |p - torch| / bound {worst:.3g}')
    # the optimizer state matches torch's too. After two steps m = 0.9 * 0.1 g1 + 0.1 g2 can cancel, so its error is
    # bounded relative to the tensor's largest value, not element by element
    sd = opt.state_dict()
    for i, n in enumerate(opt.names):
        st = torch_opt.state[rparams[n]]
        assert sd['state'][i]['step'].item() == st['step'].item() == 2
        for key in ('exp_avg', 'exp_avg_sq'):
            assert (sd['state'][i][key] - st[key]).abs().max() <= 1e-5 * st[key].abs().max(), (n, key)


def test_overflow_skips_the_step_and_backs_off():
    """fp16 build: at a scale of 2^40 the loss gradient itself (|sigmoid - label| * 2^40 / P) is far beyond 65504, the
    range check of the head's backward flags it, and the step is skipped: parameters, moments and the step count are
    bit-unchanged and the scale is halved. (A bf16 build has the fp32 exponent range, so this scale does not saturate
    it; the flag is exercised there by the kernel tests.)"""
    from vited_b200 import train
    if not _fp16():
        pytest.skip('bf16 build: 2^40 does not saturate')
    kw = _case('small_hd64')
    model, _, _ = _models(kw, 22)
    before = {n: p.detach().clone() for n, p in model.named_parameters()}
    opt = train.AdamW(model, lr=1e-3)
    scaler = train.LossScaler(init_scale=2.0 ** 40)
    out = train.train_iteration(model, _batch(kw, 6, 60), [0, 0, 0, 1, 1, 1], opt, scaler, generator=torch.Generator())
    assert out[5] is True and out[4] == math.inf
    assert scaler.scale == 2.0 ** 39 and opt.t == 0
    for n, p in model.named_parameters():
        assert torch.equal(p.detach(), before[n]), n
        assert float(opt.exp_avg[n].abs().max()) == 0.0 and float(opt.exp_avg_sq[n].abs().max()) == 0.0


def test_scale_settles_and_grows():
    """From 2^24 the scale backs off until the gradients fit (fp16 build: the first iteration overflows for certain,
    |dlogits| * 2^24 > 65504) and then steps happen; with growth_interval = 2, two clean iterations double the scale."""
    from vited_b200 import train
    kw = _case('small_hd64')
    model, _, _ = _models(kw, 23)
    opt = train.AdamW(model, lr=1e-5)
    scaler = train.LossScaler(init_scale=2.0 ** 24)
    skipped = []
    samples = _batch(kw, 6, 70)       # one batch: once the scale fits it, it keeps fitting
    for it in range(30):
        out = train.train_iteration(model, samples, [0, 0, 0, 1, 1, 1], opt, scaler,
                                    generator=torch.Generator().manual_seed(0))
        skipped.append(out[5])
    assert opt.t == skipped.count(False) and opt.t >= 8, skipped
    if _fp16():
        assert skipped[0] and scaler.scale < 2.0 ** 24
    assert not any(skipped[-8:]), skipped
    grow = train.LossScaler(init_scale=1024.0, growth_interval=2)
    for it in range(2):
        out = train.train_iteration(model, _batch(kw, 6, 90 + it), [0, 0, 0, 1, 1, 1], opt, grow,
                                    generator=torch.Generator().manual_seed(it))
        assert not out[5]
    assert grow.scale == 2048.0 and grow._growth_tracker == 0


def test_ten_iterations_track_a_float64_loop():
    """small_hd64, one fixed batch, 10 iterations at lr 1e-4 against float64: oracle autograd + clip_grad_norm_ + torch
    AdamW on float64 parameters. One step's loss agrees to 5e-3 (tests/test_gpu_train.py, 16-bit GEMM operands); each
    Adam step moves a parameter by at most ~lr whatever the gradient's rounding, so after k steps the two parameter sets
    differ by at most 2 k lr per element (2e-3 here) and the loss by that times its sensitivity; bound 2e-2 on every
    iteration's loss. Both runs must learn: the last loss is below the first. Measured on a B200 (fp16 build): the
    losses differ by at most 5.6e-5 over the 10 iterations (0.704 -> 0.165)."""
    from vited_b200 import train, synthetic
    from oracle import vited_oracle as orc
    kw = _case('small_hd64')
    model, sd = helpers.make_gpu_model(kw, 24)
    targets = [0, 0, 0, 1, 1, 1]
    samples = synthetic.synthetic_images(len(targets), kw['img_size'], seed=80)
    groups, labels = orc.train_pairs(targets, 4)
    lr = 1e-4
    opt = train.AdamW(model, lr=lr)
    scaler = train.LossScaler(init_scale=1024.0)
    p64 = {k: torch.nn.Parameter(v.double().clone()) for k, v in sd.items()}
    names = dict(model.named_parameters())
    ref = torch.optim.AdamW([{'params': [p64[n] for n in opt.groups[0]], 'weight_decay': 0.05},
                             {'params': [p64[n] for n in opt.groups[1]], 'weight_decay': 0.0}], lr=lr, foreach=False,
                            fused=False)
    ours, theirs = [], []
    for it in range(10):
        out = train.train_iteration(model, samples.cuda(), targets, opt, scaler, groups=groups, labels=labels)
        assert not out[5]
        ours.append(out[0].item())
        loss, _, _, _, grads = orc.train_step({k: p.detach() for k, p in p64.items()}, kw['num_heads'], samples.double(),
                                              targets, 4)
        for k, p in p64.items():
            p.grad = grads[k]
        torch.nn.utils.clip_grad_norm_(list(p64.values()), 5.0)
        ref.step()
        theirs.append(loss.item())
    print('losses', ours, theirs)
    assert max(abs(a - b) for a, b in zip(ours, theirs)) <= 2e-2
    assert ours[-1] < ours[0] and theirs[-1] < theirs[0]
    assert sorted(names) == sorted(p64)


def test_scoring_sees_the_updated_weights():
    """The scoring engine re-uploads its packed weights when a parameter's version changes; AdamW writes through raw
    pointers, so train_iteration bumps the versions. After an iteration, score_pairs equals a fresh model loaded from
    the updated state_dict -- and differs from the scores before the iteration."""
    import vited_b200
    from vited_b200 import train
    kw = _case('small_hd64')
    model, _, _ = _models(kw, 25)
    images = _batch(kw, 5, 100)
    pairs = torch.tensor([[0, 1], [1, 2], [3, 4], [4, 0]], dtype=torch.int64, device='cuda')
    before = model.score_pairs(images, pairs).clone()
    opt = train.AdamW(model, lr=1e-2)
    out = train.train_iteration(model, _batch(kw, 6, 101), [0, 0, 0, 1, 1, 1], opt, train.LossScaler(1024.0),
                                generator=torch.Generator())
    assert not out[5]
    after = model.score_pairs(images, pairs)
    fresh = vited_b200.VisionTransformerCustom(mlp_ratio=4., qkv_bias=True, **kw)
    fresh.load_state_dict({k: v.detach().cpu() for k, v in model.state_dict().items()})
    want = fresh.cuda().eval().score_pairs(images, pairs)
    assert torch.equal(after, want)
    assert not torch.equal(after, before)


def test_train_step_launches_no_extra_kernels():
    """train_step has no flag: the range checks and the checked attention only run inside train_iteration."""
    from vited_b200 import train
    kw = _case('small_hd64')
    model, _, _ = _models(kw, 26)
    samples = _batch(kw, 6, 110)
    train.train_step(model, samples, [0, 0, 0, 1, 1, 1], generator=torch.Generator().manual_seed(0), profile=True)
    names = set(model.train_profile)
    step_launches = model.train_launches
    assert not any('range_check' in n or 'chk' in n for n in names), names
    opt = train.AdamW(model, lr=1e-4)
    train.train_iteration(model, samples, [0, 0, 0, 1, 1, 1], opt, train.LossScaler(1024.0),
                          generator=torch.Generator().manual_seed(0))
    assert model.train_launches > step_launches
    print(f'train_step launches {step_launches}, train_iteration launches {model.train_launches}')


# ---------------------------------------------------------------------------------------------------------------
# two ranks
# ---------------------------------------------------------------------------------------------------------------
def _worker(rank, world, port, q):
    import torch.distributed as dist
    from vited_b200 import train
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group('nccl', rank=rank, world_size=world, device_id=torch.device('cuda', rank))
    try:
        out = {}
        kw = _case('small_hd64')
        targets = [0, 0, 0, 1, 1, 1]
        # rank 1's images are 3e4 times brighter: at a loss scale of 64 its patch-embedding weight gradient
        # (dY^T X over 96 patch rows) leaves the 16-bit range, rank 0's does not. Checked first on each rank alone.
        samples = _batch(kw, 6, 120 + rank) * (3e4 if rank == 1 else 1.0)
        probe, _ = helpers.make_gpu_model(kw, 27)
        res = train.train_iteration(probe, samples, targets, train.AdamW(probe, lr=1e-3), train.LossScaler(64.0),
                                    generator=torch.Generator().manual_seed(1), all_reduce=False)
        out['alone_skipped'] = res[5]
        model, _ = helpers.make_gpu_model(kw, 27)
        opt = train.AdamW(model, lr=1e-3)
        scaler = train.LossScaler(init_scale=64.0)
        res = train.train_iteration(model, samples, targets, opt, scaler, generator=torch.Generator().manual_seed(1))
        out['first_skipped'] = res[5]
        out['t_after_first'] = opt.t
        for it in range(4):
            samples = _batch(kw, 6, 130 + 2 * it + rank)
            train.train_iteration(model, samples, targets, opt, scaler, generator=torch.Generator().manual_seed(it))
        flat = torch.cat([p.detach().reshape(-1) for p in model.parameters()])
        both = [torch.empty_like(flat) for _ in range(world)]
        dist.all_gather(both, flat)
        out['equal'] = bool(torch.equal(both[0], both[1]))
        out['t'] = opt.t
        q.put((rank, out))
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs two GPUs')
def test_two_ranks_skip_together_and_stay_equal():
    import torch.multiprocessing as mp
    world = 2
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = 29600 + (os.getpid() + 977) % 2000
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    results = dict(q.get(timeout=600) for _ in range(world))
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    for rank, out in results.items():
        assert out['equal'], (rank, out)
    if _fp16():      # bf16 represents rank 1's gradients: nothing saturates, nothing is skipped
        assert results[1]['alone_skipped'] and not results[0]['alone_skipped'], results
        assert results[0]['first_skipped'] and results[1]['first_skipped'], results
    assert results[0]['first_skipped'] == results[1]['first_skipped']
    assert results[0]['t'] == results[1]['t'] >= 1
