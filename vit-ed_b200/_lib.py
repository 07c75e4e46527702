"""ctypes binding of the C-ABI in include/vited_b200.h (the only way Python reaches the CUDA kernels).

There is no CPU or PyTorch fallback: if ``lib/libvited_b200.so`` is missing or fails to load, importing this module
raises, and every compute entry point raises when it returns a non-zero status.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# VITED_LIB: path override used by tools/ to A/B differently built libraries (still the same C-ABI, still no fallback)
LIB_PATH = os.environ.get("VITED_LIB") or os.path.join(_HERE, "lib", "libvited_b200.so")


class VitedError(RuntimeError):
    pass


class Config(ctypes.Structure):
    """``vited_config`` (include/vited_b200.h) -- the constructor arguments of models/build.py:19-32."""

    _fields_ = [
        ("img_size", ctypes.c_int32),
        ("patch_size", ctypes.c_int32),
        ("in_chans", ctypes.c_int32),
        ("num_classes", ctypes.c_int32),
        ("embed_dim", ctypes.c_int32),
        ("depth", ctypes.c_int32),
        ("c_depth", ctypes.c_int32),
        ("num_heads", ctypes.c_int32),
        ("mlp_ratio", ctypes.c_float),
        ("qkv_bias", ctypes.c_int32),
    ]


GRID_ORDERED_OFFDIAG = 0
GRID_UPPER_TRI_DIAG = 1
OPT_GEMM_IMPL = 0
OPT_ATTN_IMPL = 1
OPT_CHUNK_ROWS = 2
OPT_CACHE_LAYER0 = 3
OPT_PROFILE = 4
OPT_PRUNE_TAIL = 5
OPT_FUSE_LN = 6
OPT_KV_BUDGET_MB = 7
OPT_FUSE_MLP = 8
OPT_XSRC_BUDGET_MB = 9

_vp = ctypes.c_void_p
_i = ctypes.c_int
_i64 = ctypes.c_int64
_f = ctypes.c_float
_d = ctypes.c_double

# name -> (restype, argtypes); kept in one table so tests can check it against the header
SIGNATURES = {
    "vited_last_error": (ctypes.c_char_p, []),
    "vited_create": (_i, [ctypes.POINTER(Config), _i, ctypes.POINTER(_vp)]),
    "vited_destroy": (None, [_vp]),
    "vited_set_option": (_i, [_vp, _i, _i64]),
    "vited_load_weight": (_i, [_vp, ctypes.c_char_p, _vp, _i64, _vp]),
    "vited_num_weights_expected": (_i, [_vp]),
    "vited_num_weights_loaded": (_i, [_vp]),
    "vited_weight_name": (ctypes.c_char_p, [_vp, _i]),
    "vited_encode": (_i, [_vp, _vp, _i, _vp, _vp]),
    "vited_decode": (_i, [_vp, _vp, _vp, _i, _vp, _vp]),
    "vited_forward_pairs": (_i, [_vp, _vp, _i, _vp, _vp]),
    "vited_score_grid": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _vp]),
    "vited_score_grid_u8": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _vp]),
    "vited_score_pairs": (_i, [_vp, _vp, _i, _vp, _i64, _vp, _vp]),
    "vited_score_pairs_u8": (_i, [_vp, _vp, _i, _vp, _i64, _vp, _vp]),
    "vited_profile_json": (ctypes.c_char_p, [_vp, _vp]),
    "vited_launch_count": (_i64, [_vp]),
    "vited_act_dtype": (_i, []),
    "vited_prepare_pieces": (_i, [_vp, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp]),
    "vited_normalize_u8": (_i, [_vp, _i, _i, _vp, _vp]),
    "vited_retrieval_rows": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    "vited_puzzle_tables": (_i, [_vp, _i, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "vited_workspace_bytes": (_i64, [_vp]),
    "vited_train_cast": (_i, [_vp, _vp, _i64, _f, _vp]),
    "vited_train_axpby16": (_i, [_vp, _vp, _i64, _f, _f, _vp]),
    "vited_train_axpy32": (_i, [_vp, _vp, _i64, _f, _vp]),
    "vited_train_transpose": (_i, [_vp, _i, _i, _vp, _i, _i, _i, _f, _vp]),
    "vited_train_ln_forward": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _f, _vp]),
    "vited_train_ln_backward": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _f, _vp]),
    "vited_train_gelu_forward": (_i, [_vp, _vp, _i64, _vp]),
    "vited_train_gelu_backward": (_i, [_vp, _vp, _vp, _i64, _vp]),
    "vited_train_colsum": (_i, [_vp, _vp, _i, _i, _f, _vp]),
    "vited_train_gather_rows": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "vited_train_scatter_add_rows": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _f, _vp]),
    "vited_train_attention": (_i, [_i, _vp, _i, _vp, _i, _vp, _i, _vp, _i, _vp, _vp, _i, _vp, _vp, _i, _vp, _i, _vp, _i, _i, _i,
                                   _i, _i, _i, _f, _vp]),
    "vited_train_bce_logits": (_i, [_vp, _vp, _i, _vp, _vp, _f, _vp]),
    "vited_train_range_limit": (_f, []),
    "vited_train_range_check": (_i, [_vp, _i, _i64, _f, _vp, _vp]),
    "vited_train_attention_chk": (_i, [_i, _vp, _i, _vp, _i, _vp, _i, _vp, _i, _vp, _vp, _i, _vp, _vp, _i, _vp, _i, _vp, _i, _i,
                                       _i, _i, _i, _i, _f, _vp, _vp]),
    "vited_train_grad_norm": (_i, [_vp, _i, _vp, _i, _vp, _vp]),
    "vited_train_adamw": (_i, [_vp, _i, _i64, _d, _d, _d, _d, _f, _d, _d, _vp]),
    "vited_op_gemm": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "vited_op_gemm_resid_ln": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _f, _vp]),
    "vited_op_mlp_resid_ln": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _f, _vp]),
    "vited_op_cproj_mlp_resid_ln": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _f,
                                         _vp]),
    "vited_op_resid_ln": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _f, _vp]),
    "vited_op_attention": (_i, [_vp, _i, _vp, _i, _vp, _i, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _f, _i, _vp]),
    "vited_op_attention_cls": (_i, [_vp, _i, _vp, _i, _vp, _i, _vp, _i, _i, _i, _i, _i, _i, _i, _vp, _f, _vp]),
    "vited_op_head": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _f, _vp]),
    "vited_op_im2col": (_i, [_vp, _vp, _i, _i, _i, _i, _vp]),
    "vited_op_im2col_u8": (_i, [_vp, _vp, _i, _i, _i, _i, _vp]),
}


def _load():
    if not os.path.exists(LIB_PATH):
        raise VitedError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or vit-ed_b200/csrc/build.sh). This package has no CPU / PyTorch fallback."
        )
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    return lib


lib = _load()


def act_dtype():
    """torch dtype of the 16-bit operands the single-kernel entry points take (fp16 unless built with
    -DVITED_ACT_BF16=1); ``ACT_NAME`` is the matching string for bench.py's ``dtype``."""
    import torch
    return torch.bfloat16 if lib.vited_act_dtype() == 1 else torch.float16


ACT_NAME = 'bf16' if lib.vited_act_dtype() == 1 else 'fp16'


def range_limit():
    """|x| from which a value does not survive this build's 16-bit conversion: 65504.0 (fp16, where conversions
    saturate) or inf (bf16, where only non-finite values are lost). ``vited_train_range_check`` flags values at or
    beyond it."""
    return float(lib.vited_train_range_limit())


def last_error() -> str:
    msg = lib.vited_last_error()
    return msg.decode("utf-8", "replace") if msg else ""


def check(status: int, what: str) -> None:
    if status != 0:
        raise VitedError(f"{what} failed: {last_error()}")
