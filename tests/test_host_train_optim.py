"""CPU: the host side of train.train_iteration -- LossScaler against torch.amp.GradScaler, the no-decay parameter
groups of train.AdamW on the Hisfrag20 model, and AdamW's state_dict against torch.optim.AdamW in both directions."""
import random

import pytest
import torch

from tests import helpers


def _scaler_step(ref, opt, p, found_inf):
    """one GradScaler iteration whose unscale_ finds an inf (found_inf) or only finite gradients"""
    ref.scale(torch.ones(()))
    p.grad = torch.full_like(p, float('inf') if found_inf else 1.0)
    ref.step(opt)
    ref.update()


@pytest.mark.parametrize('seed', [0, 1, 2])
def test_loss_scaler_follows_grad_scaler(seed):
    from vited_b200 import train
    rng = random.Random(seed)
    kw = dict(init_scale=2.0 ** rng.randint(4, 30), growth_interval=rng.choice([1, 2, 3, 7]))
    ref = torch.amp.GradScaler('cpu', **kw)
    ours = train.LossScaler(**kw)
    p = torch.nn.Parameter(torch.zeros(3))
    opt = torch.optim.SGD([p], lr=0.0)
    for i in range(300):
        found_inf = rng.random() < (0.5 if i < 100 else 0.05)
        _scaler_step(ref, opt, p, found_inf)
        ours.update(found_inf)
        assert ours.scale == ref.get_scale(), i
        assert ours.state_dict() == ref.state_dict(), i
    # the state dicts are interchangeable
    other = train.LossScaler()
    other.load_state_dict(ref.state_dict())
    assert other.state_dict() == ref.state_dict()
    back = torch.amp.GradScaler('cpu')
    back.load_state_dict(ours.state_dict())
    assert back.state_dict() == ours.state_dict()


def test_loss_scaler_growth_stays_finite():
    from vited_b200 import train
    s = train.LossScaler(init_scale=2.0 ** 127, growth_interval=1)
    s.update(False)
    assert s.scale == 2.0 ** 127       # 2^128 is not a float32: GradScaler keeps the old scale
    s.update(True)
    assert s.scale == 2.0 ** 126


def _hisfrag20_model():
    import vited_b200
    _, kw = helpers.load_model_case('hisfrag20_patch16_512')
    return vited_b200.VisionTransformerCustom(mlp_ratio=4., qkv_bias=True, **kw)


def test_no_decay_groups_on_the_hisfrag20_model():
    from vited_b200 import train
    model = _hisfrag20_model()
    opt = train.AdamW(model, lr=1e-3)
    decay, no_decay = map(set, opt.groups)
    names = {n for n, _ in model.named_parameters()}
    assert decay | no_decay == names and not decay & no_decay
    # every weight matrix (and the patch-embedding convolution) decays; nothing else does
    assert decay == {n for n, p in model.named_parameters() if p.dim() >= 2 and n not in ('pos_embed', 'cls_token')}
    assert {'pos_embed', 'cls_token', 'head.bias', 'norm.weight', 'norm.bias', 'blocks.0.norm1.weight',
            'blocks.0.attn.qkv.bias', 'cross_blocks.11.norm_context.bias'} <= no_decay
    assert {'patch_embed.proj.weight', 'blocks.0.attn.qkv.weight', 'cross_blocks.0.cross_attn.kv.weight',
            'head.weight'} <= decay
    assert len(decay) == 12 * 4 + 12 * 7 + 2
    assert sum(p.numel() for n, p in model.named_parameters()) > 50_000_000
    assert opt.group_decay == [0.05, 0.0]
    # an explicit set replaces the rule
    only = train.AdamW(model, lr=1e-3, no_decay={'head.bias'})
    assert only.groups[1] == ['head.bias'] and len(only.groups[0]) == len(names) - 1
    with pytest.raises(ValueError):
        train.AdamW(model, lr=1e-3, no_decay={'not_a_parameter'})


def test_adamw_state_dict_round_trips_through_torch():
    import vited_b200
    from vited_b200 import train
    _, kw = helpers.load_model_case('small_hd64')
    model = vited_b200.VisionTransformerCustom(mlp_ratio=4., qkv_bias=True, **kw)
    opt = train.AdamW(model, lr=3e-4, betas=(0.8, 0.99), eps=1e-7, weight_decay=0.1)
    fresh = opt.state_dict()
    assert fresh['state'] == {}
    g = torch.Generator().manual_seed(0)
    opt.t = 17
    for n in opt.names:
        opt.exp_avg[n].copy_(torch.randn(opt.exp_avg[n].shape, generator=g))
        opt.exp_avg_sq[n].copy_(torch.rand(opt.exp_avg_sq[n].shape, generator=g))
    sd = opt.state_dict()
    params = dict(model.named_parameters())
    ref = torch.optim.AdamW(opt._torch_groups(params), lr=1.0, foreach=False, fused=False)
    ref.load_state_dict(sd)
    rsd = ref.state_dict()
    for a, b in zip(rsd['param_groups'], sd['param_groups']):
        assert a == b
    assert rsd['param_groups'][0]['weight_decay'] == 0.1 and rsd['param_groups'][1]['weight_decay'] == 0.0
    assert rsd['param_groups'][0]['lr'] == 3e-4 and rsd['param_groups'][0]['betas'] == (0.8, 0.99)
    assert sorted(rsd['state']) == list(range(len(opt.names)))
    for i, n in enumerate(opt.names):
        assert ref.state[params[n]]['step'].item() == 17.0
        assert torch.equal(ref.state[params[n]]['exp_avg'], opt.exp_avg[n])
        assert torch.equal(ref.state[params[n]]['exp_avg_sq'], opt.exp_avg_sq[n])
    back = train.AdamW(model, lr=1.0)
    back.load_state_dict(rsd)
    assert back.t == 17 and back.lr == 3e-4 and back.betas == (0.8, 0.99) and back.eps == 1e-7
    assert back.group_decay == [0.1, 0.0]
    for n in opt.names:
        assert torch.equal(back.exp_avg[n], opt.exp_avg[n]) and torch.equal(back.exp_avg_sq[n], opt.exp_avg_sq[n])
    # a torch optimizer that never stepped has no state: moments zero, step 0
    back.load_state_dict(fresh)
    assert back.t == 0 and all(float(back.exp_avg[n].abs().max()) == 0.0 for n in back.names)
