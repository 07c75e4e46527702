"""Overhead of train.train_iteration (range checks, gradient norm, fused AdamW, one 8-byte read back) over
train.train_step on the real Hisfrag20 configuration: 24 images of 512 px from 8 writers -> 72 pairs, 12 + 12 layers.
The two calls alternate in one process on the same batch; prints the card's name and power limit with the numbers.

    python tools/train_iteration.py [--rounds 5] [--out DIR]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def _card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i', '0'],
                       capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else torch.cuda.get_device_name(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--rounds', type=int, default=5)
    ap.add_argument('--out', default=None, help='directory for the JSON result (default: print only)')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('train_iteration.py measures on a CUDA device; none found')
    import vited_b200
    from vited_b200 import synthetic, train
    model = vited_b200.build_model(vited_b200.get_config('hisfrag'))
    model.load_state_dict(synthetic.synthetic_state_dict(model, seed=0))
    model = model.cuda()
    targets = [i // 3 for i in range(24)]
    samples = synthetic.synthetic_images(24, model.img_size, seed=1).cuda()
    groups, labels = train.prepare_pairs(targets, torch.Generator().manual_seed(0))
    opt = train.AdamW(model, lr=1e-5)
    scaler = train.LossScaler(init_scale=1024.0, growth_interval=10 ** 9)   # a fixed scale: every round does the same work

    def timed(fn):
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b), out

    step = lambda: train.train_step(model, samples, targets, groups=groups, labels=labels)
    iteration = lambda: train.train_iteration(model, samples, targets, opt, scaler, groups=groups, labels=labels)
    step()
    iteration()                                                               # warm-up of both shapes
    t_step, t_iter, skipped = [], [], 0
    for _ in range(args.rounds):
        ms, _ = timed(step)
        t_step.append(ms)
        launches_step = model.train_launches
        ms, out = timed(iteration)
        t_iter.append(ms)
        skipped += int(out[5])
        launches_iter = model.train_launches
    s, i = statistics.median(t_step), statistics.median(t_iter)
    res = {'card': _card(), 'pairs': int(groups.shape[0]), 'rounds': args.rounds, 'train_step_ms': round(s, 2),
           'train_iteration_ms': round(i, 2), 'overhead_ms': round(i - s, 2), 'overhead_pct': round(100 * (i - s) / s, 2),
           'train_step_ms_all': [round(x, 2) for x in t_step], 'train_iteration_ms_all': [round(x, 2) for x in t_iter],
           'train_step_launches': launches_step, 'train_iteration_launches': launches_iter, 'skipped': skipped,
           'act': str(vited_b200._lib.ACT_NAME)}
    print(json.dumps(res))
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, 'train_iteration.json'), 'w') as f:
            json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
