"""GPU: VisionTransformerCustom under torch.autograd. In training mode, with gradients wanted, the three forward modes
are autograd Functions backed by the training kernels (train.encode / train.decode), so the reference's own training
loop -- ``tokens = model(x, forward_first_part=True); logits = model(tokens[g1], x[g0]); loss.backward()`` with
GradScaler, clip_grad_norm_, a torch optimizer, DDP -- runs unchanged. Every other call runs the scoring engine.

Bounds are in units of u, the unit roundoff of the library's 16-bit type (tests/test_gpu_train_kernels.py: _u16,
STEP_REL_L2, STEP_ELEM), or are the bounds the train_step tests use at the same size (tests/test_gpu_train.py)."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests import helpers
from tests.conftest import GOLDEN
from tests.test_gpu_train_kernels import STEP_ELEM, STEP_REL_L2, _act, _u16

pytestmark = pytest.mark.gpu

IMAGE_SEED = {'test_patch32_64': 11, 'small_hd64': 12}     # tests/golden/make_golden.py CASES, as test_gpu_train.py
# p.grad of the two-phase autograd loop against train_step's own p.grad on the same batch, relative L2 per tensor in
# units of u. The two run the same kernels; they differ in the loss scale of the 16-bit gradient operands (1 here, 1024
# in train_step: gradients below the fp16 normal range lose bits here), in the order of the atomic scatter-adds, and in
# the decoder's patch embedding (per pair here, per item there). Measured on a B200: 0.86 u (fp16 build), 0.83 u (bf16),
# at every size below.
VS_TRAIN_STEP = 4
# The loss scale of the two-phase tests: train_step's default, the scale their bounds were measured at. Without a
# scale, fp16 gradients of the deeper layers fall below the fp16 normal range at these sizes (as under fp16 autocast).
SCALE = 1024.0


def _model(kw, seed):
    model, sd = helpers.make_gpu_model(kw, seed)
    return model.train(), sd


def _rel_l2(got, want):
    got, want = got.detach().double().cpu(), want.detach().double().cpu()
    return float((got - want).norm() / max(float(want.norm()), 1e-30))


def _two_phase(model, samples, groups, labels, scale=None):
    """the reference's HisfragTrainer.train_step forward (hisfrag.py:149-159) and misc/engine.py's backward"""
    g = groups.to(samples.device)
    tokens = model(samples, forward_first_part=True)
    logits = model(tokens[g[:, 1]], samples[g[:, 0]])
    loss = F.binary_cross_entropy_with_logits(logits, labels.to(samples.device))
    (loss if scale is None else scale(loss)).backward()
    return loss.detach(), logits.detach()


def _grads(model):
    return {k: p.grad.detach().clone() for k, p in model.named_parameters()}


def _train_step_grads(kw, seed, samples, groups, labels):
    from vited_b200 import train
    ref, _ = helpers.make_gpu_model(kw, seed)
    train.train_step(ref, samples, None, groups=groups, labels=labels)
    return _grads(ref)


# ---------------------------------------------------------------------------------------------------------------
# 1. the reference's two-phase loop
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('name', ['test_patch32_64', 'small_hd64'])
def test_two_phase_loop_matches_fixture_oracle_and_train_step(name):
    """At loss scale SCALE, p.grad / SCALE within the bounds of tests/test_gpu_train.py at these sizes: gradient norms within 4e-2 and raw slices within 5e-2 of their
    max against the reference-written fixture; 5e-2 relative L2 against the oracle's float64 autograd. Against
    train_step on the same batch: VS_TRAIN_STEP u relative L2. Measured on a B200: worst 0.16 % (fp16 build) and 1.3 %
    (bf16) relative L2 against the oracle."""
    from vited_b200 import synthetic, train
    from oracle import vited_oracle as orc
    z = np.load(os.path.join(GOLDEN, 'train_step.npz'))
    zc, kw = helpers.load_model_case(name)
    model, sd = _model(kw, int(zc['weight_seed']))
    targets = z[f'{name}_targets']
    samples = synthetic.synthetic_images(len(targets), kw['img_size'], seed=IMAGE_SEED[name] + 100)
    torch.manual_seed(int(z[f'{name}_perm_seed']))
    groups, labels = train.prepare_pairs(targets)
    assert np.array_equal(labels.numpy(), z[f'{name}_labels'])
    loss, logits = _two_phase(model, samples.cuda(), groups, labels, scale=lambda l: l * SCALE)
    assert abs(loss.item() - float(z[f'{name}_loss'])) < 5e-3
    np.testing.assert_allclose(logits.cpu().numpy(), z[f'{name}_logits'], rtol=0, atol=2e-2)
    grads = {k: g / SCALE for k, g in _grads(model).items()}
    keys = [str(k) for k in z[f'{name}_grad_keys']]
    assert sorted(grads) == keys
    for k, want in zip(keys, z[f'{name}_grad_norms']):
        got = float(grads[k].double().norm())
        assert abs(got - want) / max(want, 1e-8) < 4e-2 or abs(got - want) < 1e-6, f'{k}: |grad| {got} vs {want}'
    for k in ('head.weight', 'cls_token', 'cross_blocks.0.cross_attn.kv.weight', 'blocks.0.attn.qkv.bias',
              'patch_embed.proj.weight'):
        want = z[f'{name}_grad::{k}']
        got = grads[k].flatten()[:64].cpu().numpy()
        assert np.abs(got - want).max() < 5e-2 * max(np.abs(want).max(), 1e-8), k
    o_loss, _, o_groups, _, o_grads = orc.train_step({k: v.double() for k, v in sd.items()}, kw['num_heads'],
                                                     samples.double(), targets, int(z[f'{name}_perm_seed']))
    assert torch.equal(groups, o_groups)
    ts = _train_step_grads(kw, int(zc['weight_seed']), samples.cuda(), groups, labels)
    vs_oracle = {k: _rel_l2(g, o_grads[k]) for k, g in grads.items() if float(o_grads[k].norm()) > 1e-7}
    vs_step = {k: _rel_l2(g, ts[k]) for k, g in grads.items() if float(ts[k].norm()) > 1e-7}
    u = _u16()
    print(f'[{_act()}] {name}: worst rel L2 vs float64 oracle {max(vs_oracle.values()):.3g}, '
          f'vs train_step {max(vs_step.values()):.3g} ({max(vs_step.values()) / u:.3g} u)')
    for k, e in vs_oracle.items():
        assert e < 5e-2, f'{k}: relative L2 error {e:.4f} against the oracle'
    for k, e in vs_step.items():
        assert e <= VS_TRAIN_STEP * u, f'{k}: relative L2 {e:.3g} against train_step'


def test_two_phase_loop_at_hisfrag20_token_count():
    """test_train_step_at_hisfrag20_token_count's case (img 512, patch 16, embed 384, 6 heads, depth = c_depth = 1; 6
    images of two writers, 15 pairs) through the two-phase autograd loop at loss scale SCALE, with its bounds: every gradient within
    STEP_REL_L2 u relative L2 of float64 autograd, the qkv / kv / proj weight gradients within STEP_ELEM u of their max
    element by element; and within VS_TRAIN_STEP u relative L2 of train_step's gradients on the same batch. Measured on
    a B200: 7.4 u relative L2 and 2.3 u element error (fp16 build), 18.4 u and 3.5 u (bf16), as train_step's."""
    from vited_b200 import synthetic, train
    from oracle import vited_oracle as orc
    _, kw = helpers.load_model_case('hisfrag20_patch16_512')
    kw = dict(kw, depth=1, c_depth=1)
    model, sd = _model(kw, 31)
    targets = [0, 0, 0, 1, 1, 1]
    samples = synthetic.synthetic_images(len(targets), kw['img_size'], seed=131)
    groups, labels = orc.train_pairs(targets, 9)
    assert groups.shape[0] == 15
    loss, _ = _two_phase(model, samples.cuda(), groups, labels, scale=lambda l: l * SCALE)
    grads = {k: g / SCALE for k, g in _grads(model).items()}
    o_loss, _, _, _, o_grads = orc.train_step({k: v.double() for k, v in sd.items()}, kw['num_heads'], samples.double(),
                                              targets, 9)
    ts = _train_step_grads(kw, 31, samples.cuda(), groups, labels)
    u = _u16()
    rel = {k: _rel_l2(g, o_grads[k]) for k, g in grads.items()}
    elem = {k: float((g.double().cpu() - o_grads[k]).abs().max() / o_grads[k].abs().max()) for k, g in grads.items()
            if k.endswith(('qkv.weight', 'kv.weight', 'proj.weight')) and not k.startswith('patch_embed')}
    vs_step = {k: _rel_l2(g, ts[k]) for k, g in grads.items()}
    print(f'[{_act()}] Hisfrag20 tokens: worst rel L2 vs float64 {max(rel.values()) / u:.3g} u, worst element '
          f'{max(elem.values()) / u:.3g} u, worst rel L2 vs train_step {max(vs_step.values()) / u:.3g} u')
    assert len(elem) == 6
    for k, e in rel.items():
        assert e <= STEP_REL_L2[_act()] * u, f'{k}: relative L2 error {e:.3g}'
    for k, e in elem.items():
        assert e <= STEP_ELEM * u, f'{k}: element error {e:.3g} of the max'
    for k, e in vs_step.items():
        assert e <= VS_TRAIN_STEP * u, f'{k}: relative L2 {e:.3g} against train_step'
    assert abs(loss.item() - o_loss.item()) <= 4 * u * max(1.0, o_loss.item())


# ---------------------------------------------------------------------------------------------------------------
# 2. the puzzle model, one-shot model(pairs), images that require grad, a loss that is not BCE
# ---------------------------------------------------------------------------------------------------------------
def test_puzzle_pairs_with_image_gradients():
    """The puzzle model's shape (img 64, patch 8: 64 + 1 decoder tokens, embed 384, 12 heads of 32, 4 classes) cut to
    depth = c_depth = 2, 6 stacked pairs whose images require grad, loss = (logits * w).sum() with a fixed random w.
    Every parameter gradient and the image gradient within STEP_REL_L2 u relative L2 of float64 autograd of the
    oracle's forward (the image gradient is a dgrad of the patch-embedding GEMM like any other Linear input). Measured
    on a B200: worst parameter gradient 2.5 u, images 2.2 u (fp16 build); 2.7 u and 2.3 u (bf16)."""
    from vited_b200 import synthetic
    from oracle import vited_oracle as orc
    _, kw = helpers.load_model_case('puzzle_patch8_64')
    kw = dict(kw, depth=2, c_depth=2)
    model, sd = _model(kw, 41)
    n = 6
    imgs = synthetic.synthetic_images(2 * n, kw['img_size'], seed=141).view(n, 2, 3, kw['img_size'], kw['img_size'])
    w = torch.randn(n, kw['num_classes'], generator=torch.Generator().manual_seed(5), dtype=torch.float64)
    pairs = imgs.cuda().requires_grad_(True)
    logits = model(pairs)
    assert logits.shape == (n, 4) and logits.grad_fn is not None
    (logits * w.float().cuda()).sum().backward()
    p64 = {k: v.double().requires_grad_(True) for k, v in sd.items()}
    x64 = imgs.double().requires_grad_(True)
    with torch.enable_grad():
        x1, x2 = torch.unbind(x64, 1)
        o = orc.forward_head(orc.forward_second_part(orc.forward_first_part(x1, p64, kw['num_heads']), x2, p64,
                                                     kw['num_heads']), p64)
        (o * w).sum().backward()
    u = _u16()
    rel = {k: _rel_l2(p.grad, p64[k].grad) for k, p in model.named_parameters()}
    rel['images'] = _rel_l2(pairs.grad, x64.grad)
    worst = max(rel, key=rel.get)
    print(f'[{_act()}] puzzle pairs: worst rel L2 vs float64 {rel[worst] / u:.3g} u ({worst}), images '
          f'{rel["images"] / u:.3g} u, logits {float((logits.detach().cpu().double() - o.detach()).abs().max()):.3g}')
    for k, e in rel.items():
        assert e <= STEP_REL_L2[_act()] * u, f'{k}: relative L2 error {e:.3g}'


# ---------------------------------------------------------------------------------------------------------------
# 3. accumulation
# ---------------------------------------------------------------------------------------------------------------
def test_two_backward_passes_accumulate():
    """Two forward / backward passes (two batches) leave p.grad = g1 + g2 bit for bit, g1 and g2 being what each pass
    delivered to the parameter (captured by a tensor hook)."""
    from vited_b200 import synthetic, train
    _, kw = helpers.load_model_case('small_hd64')
    model, _ = _model(kw, 51)
    seen = {k: [] for k, _ in model.named_parameters()}
    for k, p in model.named_parameters():
        p.register_hook(lambda g, k=k: seen[k].append(g.detach().clone()))
    for it in range(2):
        samples = synthetic.synthetic_images(6, kw['img_size'], seed=150 + it).cuda()
        groups, labels = train.prepare_pairs([0, 0, 0, 1, 1, 1], torch.Generator().manual_seed(it))
        _two_phase(model, samples, groups, labels)
    for k, p in model.named_parameters():
        assert len(seen[k]) == 2, k
        assert torch.equal(p.grad, seen[k][0] + seen[k][1]), k
        assert not torch.equal(seen[k][0], seen[k][1]), k


# ---------------------------------------------------------------------------------------------------------------
# 4. GradScaler, torch AdamW
# ---------------------------------------------------------------------------------------------------------------
def _fixed_batch(kw, seed, targets=(0, 0, 0, 1, 1, 1), perm_seed=4):
    from vited_b200 import synthetic
    from oracle import vited_oracle as orc
    samples = synthetic.synthetic_images(len(targets), kw['img_size'], seed=seed)
    groups, labels = orc.train_pairs(list(targets), perm_seed)
    return samples, groups, labels


def test_grad_scaler_sees_a_saturated_backward():
    """fp16 build: at a scale of 2^40 the loss gradient itself is far beyond 65504. Every p.grad holds +inf in its
    first element (the decoder's range checks flag, its gradients are marked; the inf in the token gradient trips the
    encoder's checks, and its gradients are marked too), GradScaler skips torch AdamW's step and halves the scale.
    (bf16 has the fp32 exponent range: nothing saturates at this scale.)"""
    if _act() != torch.float16:
        pytest.skip('bf16 build: 2^40 does not saturate')
    _, kw = helpers.load_model_case('small_hd64')
    model, _ = _model(kw, 52)
    before = {k: p.detach().clone() for k, p in model.named_parameters()}
    opt = torch.optim.AdamW(model.parameters(), lr=1e-3)
    scaler = torch.amp.GradScaler('cuda', init_scale=2.0 ** 40)
    samples, groups, labels = _fixed_batch(kw, 160)
    _two_phase(model, samples.cuda(), groups, labels, scale=scaler.scale)
    for k, p in model.named_parameters():
        assert torch.isinf(p.grad.view(-1)[0]), k
    scaler.step(opt)
    scaler.update()
    assert scaler.get_scale() == 2.0 ** 39
    for k, p in model.named_parameters():
        assert torch.equal(p.detach(), before[k]), k


def test_grad_scale_carries_into_p_grad():
    """At scale 1024 every gradient is finite and equals 1024 x the scale-1 gradient up to the rounding of its 16-bit
    operands (a power-of-two scale is exact except where scale-1 gradients fall below the fp16 normal range) and the
    order of the atomic adds: 8 u relative L2 per tensor. Measured on a B200: 2.5 u (fp16 build, from the scale-1
    underflow), 4e-5 u (bf16, atomics only)."""
    _, kw = helpers.load_model_case('small_hd64')
    model, _ = _model(kw, 53)
    samples, groups, labels = _fixed_batch(kw, 161)
    _two_phase(model, samples.cuda(), groups, labels)
    g1 = _grads(model)
    model.zero_grad(set_to_none=True)
    scaler = torch.amp.GradScaler('cuda', init_scale=1024.0)
    _two_phase(model, samples.cuda(), groups, labels, scale=scaler.scale)
    u = _u16()
    worst = 0.0
    for k, p in model.named_parameters():
        assert torch.isfinite(p.grad).all(), k
        e = _rel_l2(p.grad / 1024.0, g1[k])
        worst = max(worst, e)
        assert e <= 8 * u, f'{k}: {e:.3g}'
    print(f'[{_act()}] scale 1024 vs scale 1: worst relative L2 {worst:.3g} ({worst / u:.3g} u)')


def test_ten_iterations_with_grad_scaler_track_a_float64_loop():
    """test_ten_iterations_track_a_float64_loop with the reference's loop instead of train_iteration: the two-phase
    calls, BCE, GradScaler (init 1024), unscale_, clip_grad_norm_(5.0), torch AdamW with the decay / no-decay groups,
    against oracle autograd + clip_grad_norm_ + torch AdamW on float64 parameters. Its bound: every iteration's loss
    within 2e-2; both runs learn."""
    from vited_b200 import train
    from oracle import vited_oracle as orc
    _, kw = helpers.load_model_case('small_hd64')
    model, sd = _model(kw, 24)
    targets = [0, 0, 0, 1, 1, 1]
    samples, groups, labels = _fixed_batch(kw, 80, targets)
    lr = 1e-4
    named = dict(model.named_parameters())
    decay = [n for n, p in named.items() if not train.default_no_decay(n, p)]
    no_decay = [n for n, p in named.items() if train.default_no_decay(n, p)]
    opt = torch.optim.AdamW([{'params': [named[n] for n in decay], 'weight_decay': 0.05},
                             {'params': [named[n] for n in no_decay], 'weight_decay': 0.0}], lr=lr)
    scaler = torch.amp.GradScaler('cuda', init_scale=1024.0)
    p64 = {k: torch.nn.Parameter(v.double().clone()) for k, v in sd.items()}
    ref = torch.optim.AdamW([{'params': [p64[n] for n in decay], 'weight_decay': 0.05},
                             {'params': [p64[n] for n in no_decay], 'weight_decay': 0.0}], lr=lr, foreach=False,
                            fused=False)
    ours, theirs = [], []
    for it in range(10):
        opt.zero_grad(set_to_none=True)
        loss, _ = _two_phase(model, samples.cuda(), groups, labels, scale=scaler.scale)
        scaler.unscale_(opt)
        torch.nn.utils.clip_grad_norm_(model.parameters(), 5.0)
        scaler.step(opt)
        scaler.update()
        assert scaler.get_scale() == 1024.0          # no step was skipped
        ours.append(loss.item())
        o_loss, _, _, _, grads = orc.train_step({k: p.detach() for k, p in p64.items()}, kw['num_heads'],
                                                samples.double(), targets, 4)
        for k, p in p64.items():
            p.grad = grads[k]
        torch.nn.utils.clip_grad_norm_(list(p64.values()), 5.0)
        ref.step()
        theirs.append(o_loss.item())
    print('losses', ours, theirs)
    assert max(abs(a - b) for a, b in zip(ours, theirs)) <= 2e-2
    assert ours[-1] < ours[0] and theirs[-1] < theirs[0]


# ---------------------------------------------------------------------------------------------------------------
# 5. scoring is unchanged
# ---------------------------------------------------------------------------------------------------------------
def test_which_path_a_forward_takes():
    """Differentiable only with grad mode on, the module in training mode and something requiring grad."""
    from vited_b200 import synthetic
    _, kw = helpers.load_model_case('small_hd64')
    model, _ = _model(kw, 54)
    x = synthetic.synthetic_images(4, kw['img_size'], seed=170).cuda()
    assert model(x, forward_first_part=True).grad_fn is not None
    with torch.no_grad():
        assert model(x, forward_first_part=True).grad_fn is None
    with torch.inference_mode():
        assert not model(x, forward_first_part=True).requires_grad
    model.eval()
    assert model(x, forward_first_part=True).grad_fn is None
    model.train()
    model.requires_grad_(False)
    tokens = model(x, forward_first_part=True)
    assert tokens.grad_fn is None
    assert model(tokens, x).grad_fn is None
    assert model(torch.stack([x, x], 1)).grad_fn is None
    assert model(tokens.requires_grad_(True), x).grad_fn is not None      # a floating-point input that requires grad
    xg = x.clone().requires_grad_(True)
    assert model(xg, forward_first_part=True).grad_fn is not None
    model.cross_blocks[0].requires_grad_(True)                            # a decoder parameter only
    assert model(x, forward_first_part=True).grad_fn is None
    assert model(tokens.detach(), x).grad_fn is not None


def test_training_calls_leave_scoring_bit_identical():
    """A model that went through training-mode forward / backward calls scores, in eval() and under no_grad, exactly as
    a fresh eval() model with the same weights, with the same number of engine launches."""
    from vited_b200 import synthetic
    _, kw = helpers.load_model_case('small_hd64')
    model, sd = _model(kw, 55)
    samples, groups, labels = _fixed_batch(kw, 171)
    _two_phase(model, samples.cuda(), groups, labels)
    fresh, _ = helpers.make_gpu_model(kw, 55)
    pairs = synthetic.synthetic_images(10, kw['img_size'], seed=172).view(5, 2, 3, kw['img_size'], kw['img_size']).cuda()
    assert model.launch_count() == fresh.launch_count() == 0              # training calls leave the engine alone
    with torch.no_grad():
        got = model(pairs)                                                # training mode under no_grad
    want = fresh(pairs)
    assert torch.equal(got, want)
    assert model.launch_count() == fresh.launch_count() > 0
    model.eval()
    n0, f0 = model.launch_count(), fresh.launch_count()
    assert torch.equal(model(pairs), fresh(pairs))
    assert model.launch_count() - n0 == fresh.launch_count() - f0 > 0
    tok_a, tok_b = model(pairs[:, 0], forward_first_part=True), fresh(pairs[:, 0], forward_first_part=True)
    assert torch.equal(tok_a, tok_b)
    assert torch.equal(model(tok_a, pairs[:, 1]), fresh(tok_b, pairs[:, 1]))


def test_scoring_sees_the_weights_after_optimizer_step():
    import vited_b200
    _, kw = helpers.load_model_case('small_hd64')
    model, _ = _model(kw, 56)
    images = _fixed_batch(kw, 173)[0].cuda()
    pairs = torch.tensor([[0, 1], [1, 2], [3, 4], [4, 0]], dtype=torch.int64, device='cuda')
    before = model.score_pairs(images, pairs).clone()
    opt = torch.optim.AdamW(model.parameters(), lr=1e-2)
    samples, groups, labels = _fixed_batch(kw, 174)
    _two_phase(model, samples.cuda(), groups, labels)
    opt.step()
    after = model.score_pairs(images, pairs)
    fresh = vited_b200.VisionTransformerCustom(mlp_ratio=4., qkv_bias=True, **kw)
    fresh.load_state_dict({k: v.detach().cpu() for k, v in model.state_dict().items()})
    assert torch.equal(after, fresh.cuda().eval().score_pairs(images, pairs))
    assert not torch.equal(after, before)


def test_backward_frees_the_saved_activations():
    """After backward (and the caller dropping its outputs), the allocator holds what it held before the forward plus
    the gradients: one 512-byte-rounded block per parameter."""
    _, kw = helpers.load_model_case('small_hd64')
    model, _ = _model(kw, 57)
    samples, groups, labels = _fixed_batch(kw, 175)
    samples = samples.cuda()
    g = groups.cuda()
    y = labels.cuda()
    torch.cuda.synchronize()
    before = torch.cuda.memory_allocated()
    tokens = model(samples, forward_first_part=True)
    logits = model(tokens[g[:, 1]], samples[g[:, 0]])
    loss = F.binary_cross_entropy_with_logits(logits, y)
    during = torch.cuda.memory_allocated()
    loss.backward()
    del tokens, logits, loss
    torch.cuda.synchronize()
    grads = sum((p.numel() * 4 + 511) // 512 * 512 for p in model.parameters())
    print(f'allocated: before {before}, after forward {during}, after backward {torch.cuda.memory_allocated()}, '
          f'gradients {grads}')
    assert during > before + grads
    assert torch.cuda.memory_allocated() == before + grads


# ---------------------------------------------------------------------------------------------------------------
# 6. errors
# ---------------------------------------------------------------------------------------------------------------
def test_cpu_inputs_still_raise():
    import vited_b200
    _, kw = helpers.load_model_case('small_hd64')
    model, _ = _model(kw, 58)
    s = kw['img_size']
    x = torch.zeros(2, 3, s, s, requires_grad=True)
    with pytest.raises(vited_b200.VitedError):
        model(x, forward_first_part=True)
    with pytest.raises(vited_b200.VitedError):
        model(torch.zeros(2, 16, kw['embed_dim']), x)
    with pytest.raises(vited_b200.VitedError):
        model(torch.zeros(2, 2, 3, s, s, requires_grad=True))
    with pytest.raises(ValueError):
        model(torch.zeros(2, 3, s + 8, s + 8, device='cuda'), forward_first_part=True)


def test_double_backward_raises():
    _, kw = helpers.load_model_case('small_hd64')
    model, _ = _model(kw, 59)
    samples, groups, labels = _fixed_batch(kw, 176)
    with pytest.raises(RuntimeError, match='double backward'):
        _two_phase(model, samples.cuda(), groups, labels, scale=lambda l: _CreateGraph(l))


class _CreateGraph:
    def __init__(self, loss):
        self.loss = loss

    def backward(self):
        self.loss.backward(create_graph=True)


def test_second_backward_through_a_retained_graph_raises():
    """backward(retain_graph=True) twice: the second raises (the activations were freed by the first) and leaves the
    gradients of the first."""
    _, kw = helpers.load_model_case('small_hd64')
    model, _ = _model(kw, 60)
    samples, groups, labels = _fixed_batch(kw, 177)
    samples, g = samples.cuda(), groups.cuda()
    tokens = model(samples, forward_first_part=True)
    loss = F.binary_cross_entropy_with_logits(model(tokens[g[:, 1]], samples[g[:, 0]]), labels.cuda())
    loss.backward(retain_graph=True)
    first = _grads(model)
    with pytest.raises(RuntimeError, match='freed'):
        loss.backward(retain_graph=True)
    for k, p in model.named_parameters():
        assert torch.equal(p.grad, first[k]), k
    with pytest.raises(RuntimeError):
        loss.backward()


# ---------------------------------------------------------------------------------------------------------------
# 7. DistributedDataParallel
# ---------------------------------------------------------------------------------------------------------------
def _ddp_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group('nccl', rank=rank, world_size=world, device_id=torch.device('cuda', rank))
    try:
        _, kw = helpers.load_model_case('small_hd64')
        batches = [_fixed_batch(kw, 180 + r) for r in range(world)]
        alone = []
        for r in range(world):                       # every rank's batch without DDP, on this rank
            m, _ = _model(kw, 61)
            _two_phase(m, batches[r][0].cuda(), batches[r][1], batches[r][2])
            alone.append(_grads(m))
        model, _ = _model(kw, 61)
        ddp = torch.nn.parallel.DistributedDataParallel(model, device_ids=[rank])
        samples, groups, labels = batches[rank]
        _two_phase(ddp, samples.cuda(), groups, labels)
        worst = 0.0
        for k, p in model.named_parameters():
            want = sum(a[k] for a in alone) / world
            worst = max(worst, _rel_l2(p.grad, want))
        q.put((rank, worst))
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs two GPUs')
def test_ddp_gradients_are_the_mean_of_the_ranks():
    import torch.multiprocessing as mp
    world = 2
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = 29600 + (os.getpid() + 1313) % 2000
    procs = [ctx.Process(target=_ddp_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    results = dict(q.get(timeout=600) for _ in range(world))
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    print(f'DDP: worst relative L2 of p.grad against the mean of the ranks\' gradients: {results}')
    assert all(w <= 1e-6 for w in results.values()), results
