"""GPU box, one GPU, one call: caller-given pair lists against the dense grid paths, and the extension of a scored
fragment collection against its full re-score.

Arms (synthetic weights of the real model shapes, random uint8 crops / fp32 pieces drawn from a seed):
  hisfrag_dense   Hisfrag20 model, 512 fragments: grid.score_fragments (vited_score_grid, upper triangle) against
                  grid.score_pairs(upper_tri_pairs(512)) (vited_score_pairs), alternating, --reps times each
  puzzle_dense    puzzle model, 540 pieces: score_grid(ORDERED_OFFDIAG) against the same ordered pairs as a list,
                  alternating, --reps times each
  extension       Hisfrag20 model, 2,048 old + 64 new fragments (new ones at evenly spread sorted positions):
                  grid.extend_fragments against grid.score_fragments of all 2,112, once each
Every shape is warmed up first. Times are synchronised wall clock around each call. The largest output difference
between the two forms of an arm is reported (0 expected for the dense arms: same chunks by construction). The card's
name, power limit and maximum SM clock come from nvidia-smi in the same call. One JSON line per arm goes to
OUT_DIR/pair_lists.jsonl.

usage: python tools/pair_lists.py OUT_DIR [--reps 2] [--arms hisfrag_dense,puzzle_dense,extension]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import vited_b200  # noqa: E402
from vited_b200 import grid, synthetic  # noqa: E402


def crops_u8(n, s, seed):
    g = torch.Generator(device='cuda').manual_seed(seed)
    return torch.randint(0, 256, (n, s, s, 3), generator=g, device='cuda', dtype=torch.int16).to(torch.uint8)


def model_for(name):
    model = vited_b200.build_model(vited_b200.get_config(name))
    model.load_state_dict(synthetic.synthetic_state_dict(model, seed=0), strict=True)
    return model.cuda().eval()


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, time.perf_counter() - t0


def ab(name_a, fn_a, name_b, fn_b, reps):
    """alternating runs; returns (per-arm seconds lists, last outputs)"""
    secs = {name_a: [], name_b: []}
    outs = {}
    for _ in range(reps):
        for name, fn in ((name_a, fn_a), (name_b, fn_b)):
            outs[name], t = timed(fn)
            secs[name].append(round(t, 4))
    return secs, outs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('out_dir')
    ap.add_argument('--reps', type=int, default=2)
    ap.add_argument('--arms', default='hisfrag_dense,puzzle_dense,extension')
    args = ap.parse_args()
    os.makedirs(args.out_dir, exist_ok=True)
    smi = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                         capture_output=True, text=True).stdout.strip().splitlines()
    gpu = smi[0] if smi else 'unknown'
    print('gpu:', gpu, flush=True)
    arms = args.arms.split(',')
    path = os.path.join(args.out_dir, 'pair_lists.jsonl')
    with open(path, 'w') as f:
        def emit(rec):
            rec['gpu'] = gpu
            print(json.dumps(rec), flush=True)
            f.write(json.dumps(rec) + '\n')
            f.flush()

        if 'hisfrag_dense' in arms or 'extension' in arms:
            his = model_for('hisfrag')
            warm = crops_u8(6, 512, 1)
            grid.score_fragments(his, warm)
            his.score_pairs(warm, torch.from_numpy(grid.upper_tri_pairs(6)).cuda())
            torch.cuda.synchronize()
        if 'hisfrag_dense' in arms:
            n = 512
            images = crops_u8(n, 512, 1234)
            pairs = torch.from_numpy(grid.upper_tri_pairs(n)).cuda()
            secs, outs = ab('grid', lambda: grid.score_fragments(his, images),
                            'pairs', lambda: grid.score_pairs(his, images, pairs), args.reps)
            p = pairs.long()
            diff = (outs['pairs'][:, 0] - outs['grid'][p[:, 0], p[:, 1]]).abs().max().item()
            emit({'arm': 'hisfrag_dense', 'n': n, 'pairs': len(pairs), 'seconds': secs,
                  'pairs_over_grid_median': round(float(np.median(secs['pairs']) / np.median(secs['grid'])), 4),
                  'max_abs_diff': diff})
            del images, outs
        if 'puzzle_dense' in arms:
            puz = model_for('puzzle')
            n = 540
            images = synthetic.synthetic_images(n, 64, seed=7).cuda()
            pairs = torch.from_numpy(grid.ordered_pairs(n)).cuda()
            puz.score_grid(images[:16], vited_b200.GRID_ORDERED_OFFDIAG)
            puz.score_pairs(images[:16], torch.from_numpy(grid.ordered_pairs(16)).cuda())
            puz.score_grid(images, vited_b200.GRID_ORDERED_OFFDIAG)
            puz.score_pairs(images, pairs)
            secs, outs = ab('grid', lambda: puz.score_grid(images, vited_b200.GRID_ORDERED_OFFDIAG),
                            'pairs', lambda: puz.score_pairs(images, pairs), max(args.reps, 3))
            p = pairs.long()
            diff = (outs['pairs'] - outs['grid'][p[:, 0], p[:, 1]]).abs().max().item()
            emit({'arm': 'puzzle_dense', 'n': n, 'pairs': len(pairs), 'seconds': secs,
                  'pairs_over_grid_median': round(float(np.median(secs['pairs']) / np.median(secs['grid'])), 4),
                  'max_abs_diff': diff})
            del images, outs
        if 'extension' in arms:
            n_old, n_new = 2048, 64
            n = n_old + n_new
            images = crops_u8(n, 512, 4321)
            is_new = np.zeros(n, dtype=bool)
            is_new[np.linspace(0, n - 1, n_new).round().astype(int)] = True
            old = torch.from_numpy(np.flatnonzero(~is_new)).cuda()
            full, t_full = timed(lambda: grid.score_fragments(his, images))
            old_sim = full[old[:, None], old[None, :]].clone()     # the old items' matrix, as a previous call left it
            ext, t_ext = timed(lambda: grid.extend_fragments(his, images, old_sim, is_new))
            n_pairs = len(grid.extension_pairs(is_new))
            emit({'arm': 'extension', 'n_old': n_old, 'n_new': n_new, 'extension_pairs': n_pairs,
                  'rescore_pairs': n * (n + 1) // 2, 'pair_ratio': round(n * (n + 1) / 2 / n_pairs, 2),
                  'seconds_rescore': round(t_full, 3), 'seconds_extension': round(t_ext, 3),
                  'time_ratio': round(t_full / t_ext, 2), 'max_abs_diff': (ext - full).abs().max().item()})


if __name__ == '__main__':
    main()
