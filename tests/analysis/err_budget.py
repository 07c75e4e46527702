"""GPU: max |logit - fp32 oracle| of the puzzle model on a small grid under different engine options (which kernel
choices contribute to the error budget of 2e-2)."""
import os, sys
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import vited_b200
from vited_b200 import grid, synthetic
from oracle import vited_oracle as orc

for seed in (0, 5):
    model = vited_b200.build_model(vited_b200.get_config('puzzle'))
    sd = synthetic.synthetic_state_dict(model, seed=seed)
    model.load_state_dict(sd, strict=True)
    model = model.cuda().eval()
    images = synthetic.synthetic_images(int(os.environ.get('N_ITEMS', '16')), 64, seed=33)
    want = orc.score_puzzle_grid(sd, 12, images, batch=80)
    small = {vited_b200.OPT_CHUNK_ROWS: 65 * 100}   # chunks of 6,500 rows take the unfused residual + LayerNorm path
    for name, opts in (('default', {}), ('unfused LN', small), ('mma.sync attention', {vited_b200.OPT_ATTN_IMPL: 2}),
                       ('unfused + mma.sync', {**small, vited_b200.OPT_ATTN_IMPL: 2})):
        model.set_option(vited_b200.OPT_CHUNK_ROWS, 524288)
        model.set_option(vited_b200.OPT_ATTN_IMPL, 0)
        for k, v in opts.items():
            model.set_option(k, v)
        got = grid.score_puzzle(model, images.cuda()).cpu()
        err = (got - want).abs()
        off = ~torch.eye(got.shape[0], dtype=torch.bool)
        agree = (got.argmax(-1) == want.argmax(-1))[off].float().mean().item()
        top2 = want.topk(2, dim=-1).values
        close = ((top2[..., 0] - top2[..., 1]) <= 2 * err.max().item())[off].float().mean().item()
        print(f'[{vited_b200.ACT_NAME}] weights seed {seed}  {name:34s} max err {err.max().item():.5f}  mean err {err.mean().item():.5f}  '
              f'argmax agreement {agree:.4f}  (pairs whose fp32 top-2 margin is within 2 x max err: {close:.4f})')
