"""GPU box, one GPU, one call: the Hisfrag fragment grid at dataset scale (20,000 and 40,000 fragments).

Arms, each scoring about 160 k pairs (the first rows of the upper-triangular grid):
  A  20,000 fragments, fp32 images [N, 3, 512, 512], default column-state budget, rows [0, 8)
  B  20,000 fragments, uint8 crops [N, 512, 512, 3], default budget,                rows [0, 8)
  C  20,000 fragments, uint8 crops, OPT_XSRC_BUDGET_MB 8000 (4 column windows),     rows [0, 8)
  D  40,000 fragments, uint8 crops, default budget (2 column windows),              rows [0, 4)
The fragments are random bytes drawn on the device from a seed (A's floats are vited_normalize_u8 of B's bytes); the
model is Hisfrag20-shaped (patch 16, 512 px, 12 + 12 layers, embed 384) with synthetic weights. Every arm gets a fresh
engine, so its workspace is its own. Per arm: synchronised wall time of the score_grid call, torch allocator peak +
vited_workspace_bytes, the drop of cudaMemGetInfo's free bytes over the arm, and max |A - B|, max |A - C|. One JSON
line per arm goes to OUT_DIR/fragment_scale.jsonl (fp32 is not attempted at 40,000: 126 GB of images alone).

usage: python tools/fragment_scale.py OUT_DIR [--n 20000] [--n-big 40000] [--arms ABCD]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import vited_b200  # noqa: E402
from vited_b200 import _lib, synthetic  # noqa: E402

S = 512


def fragments_u8(n, seed):
    g = torch.Generator(device='cuda').manual_seed(seed)
    out = torch.empty((n, S, S, 3), dtype=torch.uint8, device='cuda')
    step = 1024
    for i in range(0, n, step):                    # bounded temporaries: randint draws int64
        k = min(step, n - i)
        out[i:i + k] = torch.randint(0, 256, (k, S, S, 3), generator=g, device='cuda', dtype=torch.int16).to(torch.uint8)
    return out


def normalize(u8):
    import ctypes
    out = torch.empty((u8.shape[0], 3, S, S), dtype=torch.float32, device='cuda')
    _lib.check(_lib.lib.vited_normalize_u8(ctypes.c_void_p(u8.data_ptr()), u8.shape[0], S, ctypes.c_void_p(out.data_ptr()),
                                           ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)), 'vited_normalize_u8')
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('out_dir')
    ap.add_argument('--n', type=int, default=20000)
    ap.add_argument('--n-big', type=int, default=40000)
    ap.add_argument('--arms', default='ABCD')
    args = ap.parse_args()
    os.makedirs(args.out_dir, exist_ok=True)
    smi = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                         capture_output=True, text=True).stdout.strip().splitlines()
    gpu = smi[0] if smi else 'unknown'
    print('gpu:', gpu, flush=True)

    model = vited_b200.build_model(vited_b200.get_config('hisfrag'))
    model.load_state_dict(synthetic.synthetic_state_dict(model, seed=0), strict=True)
    model = model.cuda().eval()
    # warm-up: module load and every kernel shape class once, on a small grid
    warm = fragments_u8(16, 1)
    model.score_grid(warm, vited_b200.GRID_UPPER_TRI_DIAG)
    model.score_grid(normalize(warm), vited_b200.GRID_UPPER_TRI_DIAG)
    del warm
    torch.cuda.synchronize()

    arms = {'A': (args.n, 'fp32', None, 8), 'B': (args.n, 'u8', None, 8), 'C': (args.n, 'u8', 8000, 8),
            'D': (args.n_big, 'u8', None, 4)}
    results = {}
    path = os.path.join(args.out_dir, 'fragment_scale.jsonl')
    with open(path, 'w') as f:
        for name in args.arms:
            n, fmt, budget, rows = arms[name]
            model._release_engine()
            torch.cuda.empty_cache()
            free0 = torch.cuda.mem_get_info()[0]
            torch.cuda.reset_peak_memory_stats()
            images = fragments_u8(n, 1234)
            if fmt == 'fp32':
                u8, images = images, None
                images = normalize(u8)
                del u8
            torch.cuda.synchronize()
            torch.cuda.empty_cache()
            torch.cuda.reset_peak_memory_stats()
            model.set_option(vited_b200.OPT_XSRC_BUDGET_MB, budget if budget else 32000)
            n0 = model.launch_count()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out = model.score_grid(images, vited_b200.GRID_UPPER_TRI_DIAG, 0, rows)
            torch.cuda.synchronize()
            secs = time.perf_counter() - t0
            free1 = torch.cuda.mem_get_info()[0]
            ws = int(_lib.lib.vited_workspace_bytes(model._engine))
            pairs = rows * n - rows * (rows - 1) // 2
            rec = {'arm': name, 'n': n, 'images': fmt, 'xsrc_budget_mb': budget or 32000, 'rows': [0, rows],
                   'pairs': pairs, 'seconds': round(secs, 3), 'pairs_per_s': round(pairs / secs, 1),
                   'launches': model.launch_count() - n0,
                   'image_bytes': images.numel() * images.element_size(),
                   'torch_peak_bytes': torch.cuda.max_memory_allocated(), 'workspace_bytes': ws,
                   'peak_bytes': torch.cuda.max_memory_allocated() + ws, 'mem_get_info_delta_bytes': free0 - free1,
                   'finite': bool(torch.isfinite(out).all()), 'gpu': gpu}
            results[name] = out[..., 0].clone()
            if 'A' in results and name in 'BC':
                rec['max_abs_vs_A'] = (results[name] - results['A']).abs().max().item()
                rec['equal_to_A'] = bool(torch.equal(results[name], results['A']))
            print(json.dumps(rec), flush=True)
            f.write(json.dumps(rec) + '\n')
            f.flush()
            del images, out
    model._release_engine()


if __name__ == '__main__':
    main()
