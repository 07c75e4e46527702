"""vit-ed_b200: B200-native all-pairs compatibility scoring for ViT-ED (glmanhtu/vit-ed), hot path only.

``import vited_b200`` (alias module at the repo root) or add this directory's parent to sys.path.
Requires the in-tree CUDA library (``lib/libvited_b200.so``, built by ``__graft_entry__.build()``); there is no
CPU fallback.
"""
from . import _lib
from ._lib import VitedError, GRID_ORDERED_OFFDIAG, GRID_UPPER_TRI_DIAG, OPT_GEMM_IMPL, OPT_ATTN_IMPL, OPT_CHUNK_ROWS, \
    OPT_CACHE_LAYER0, OPT_PROFILE, OPT_PRUNE_TAIL, OPT_FUSE_LN, OPT_KV_BUDGET_MB, OPT_FUSE_MLP, OPT_XSRC_BUDGET_MB, \
    ACT_NAME, act_dtype
from .model import VisionTransformerCustom, build_model
from .configs import get_config
from . import grid, pieces, solver_tables, synthetic, train

__all__ = [
    'VisionTransformerCustom', 'build_model', 'get_config', 'grid', 'pieces', 'solver_tables', 'synthetic', 'train', 'VitedError',
    'GRID_ORDERED_OFFDIAG', 'GRID_UPPER_TRI_DIAG', 'OPT_GEMM_IMPL', 'OPT_ATTN_IMPL', 'OPT_CHUNK_ROWS',
    'OPT_CACHE_LAYER0', 'OPT_PROFILE', 'OPT_PRUNE_TAIL', 'OPT_FUSE_LN', 'OPT_KV_BUDGET_MB', 'OPT_FUSE_MLP', 'OPT_XSRC_BUDGET_MB',
    'ACT_NAME', 'act_dtype',
]
