"""Cost of the reference-shaped training loop through torch.autograd against the closed fused form, on the real
Hisfrag20 configuration: 24 images of 512 px from 8 writers -> 72 pairs, 12 + 12 layers, one GPU.

  fused     train.train_iteration (train.AdamW, train.LossScaler)
  autograd  tokens = model(x, forward_first_part=True); logits = model(tokens[g1], x[g0]); BCE; GradScaler.scale(loss)
            .backward(); unscale_; clip_grad_norm_(5.0); torch.optim.AdamW step; GradScaler.update()

The two alternate in one process on the same batch and pairs (both at a fixed loss scale of 1024). Per loop: median ms
per iteration (CUDA events), GPU activities per iteration (kernels, copies and memsets in a torch.profiler trace of one
untimed iteration) and peak allocated memory; printed with the card's name and power limit.

    python tools/autograd_step.py [--rounds 5] [--out DIR]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def _card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i', '0'],
                       capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else torch.cuda.get_device_name(0)


def _gpu_activities(fn):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return sum(1 for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--rounds', type=int, default=5)
    ap.add_argument('--out', default=None, help='directory for the JSON result (default: print only)')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('autograd_step.py measures on a CUDA device; none found')
    import vited_b200
    from vited_b200 import synthetic, train
    model = vited_b200.build_model(vited_b200.get_config('hisfrag'))
    model.load_state_dict(synthetic.synthetic_state_dict(model, seed=0))
    model = model.cuda().train()
    targets = [i // 3 for i in range(24)]
    samples = synthetic.synthetic_images(24, model.img_size, seed=1).cuda()
    groups, labels = train.prepare_pairs(targets, torch.Generator().manual_seed(0))
    g, y = groups.cuda(), labels.cuda()
    lr = 1e-5
    opt = train.AdamW(model, lr=lr)
    scaler = train.LossScaler(init_scale=1024.0, growth_interval=10 ** 9)
    named = dict(model.named_parameters())
    t_opt = torch.optim.AdamW([{'params': [p for n, p in named.items() if not train.default_no_decay(n, p)],
                                'weight_decay': 0.05},
                               {'params': [p for n, p in named.items() if train.default_no_decay(n, p)],
                                'weight_decay': 0.0}], lr=lr)
    t_scaler = torch.amp.GradScaler('cuda', init_scale=1024.0, growth_interval=10 ** 9)

    def fused():
        return train.train_iteration(model, samples, targets, opt, scaler, groups=groups, labels=labels)[5]

    def autograd():
        t_opt.zero_grad(set_to_none=True)
        tokens = model(samples, forward_first_part=True)
        logits = model(tokens[g[:, 1]], samples[g[:, 0]])
        loss = F.binary_cross_entropy_with_logits(logits, y)
        t_scaler.scale(loss).backward()
        t_scaler.unscale_(t_opt)
        torch.nn.utils.clip_grad_norm_(model.parameters(), 5.0)
        t_scaler.step(t_opt)
        t_scaler.update()
        return t_scaler.get_scale() < 1024.0

    def timed(fn):
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        skipped = fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b), torch.cuda.max_memory_allocated() - base, skipped

    fused()
    autograd()                                                                # warm-up of both
    res = {'fused': {'ms': [], 'peak_extra_mb': [], 'skipped': 0}, 'autograd': {'ms': [], 'peak_extra_mb': [], 'skipped': 0}}
    for _ in range(args.rounds):
        for name, fn in (('fused', fused), ('autograd', autograd)):
            ms, peak, skipped = timed(fn)
            res[name]['ms'].append(round(ms, 2))
            res[name]['peak_extra_mb'].append(round(peak / 2 ** 20, 1))
            res[name]['skipped'] += int(skipped)
    for name, fn in (('fused', fused), ('autograd', autograd)):
        r = res[name]
        r['median_ms'] = round(statistics.median(r['ms']), 2)
        r['peak_extra_mb'] = max(r['peak_extra_mb'])
        r['gpu_activities'] = _gpu_activities(fn)
    f, a = res['fused']['median_ms'], res['autograd']['median_ms']
    out = {'card': _card(), 'act': vited_b200.ACT_NAME, 'pairs': int(groups.shape[0]), 'rounds': args.rounds,
           'gap_pct': round(100 * (a - f) / f, 2), **res,
           'resident_mb': round(torch.cuda.memory_allocated() / 2 ** 20, 1)}
    print(json.dumps(out))
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, 'autograd_step.json'), 'w') as fh:
            json.dump(out, fh, indent=1)


if __name__ == '__main__':
    main()
