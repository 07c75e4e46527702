"""Host-side mirror of the reference model API on top of the C-ABI engine.

Same constructor arguments, same three-mode ``forward`` and same ``state_dict`` key set / tensor shapes as
``VisionTransformerCustom`` (reference models/vision_transformer.py:275-420) and ``build_model`` (reference
models/build.py:15-32), so ``load_pretrained`` (misc/utils.py:48-127) and the callers at evaluation.py:107,
hisfrag.py:214,229 work unchanged. The parameters are ordinary fp32 ``nn.Parameter``s (that is what a checkpoint
restores); the arithmetic runs in the sm_100a kernels behind ``include/vited_b200.h``. There is no PyTorch compute
path: a forward on a non-CUDA tensor, or without the built library, raises. In training mode with gradients wanted the
forward modes are torch.autograd Functions on the training kernels (``train.encode`` / ``train.decode``), so the
reference's training loop works unchanged; see ``forward``.
"""
import ctypes
import math
from functools import partial

import torch
import torch.nn as nn

from . import _lib, train


class _PatchEmbed(nn.Module):
    """timm.layers.PatchEmbed parameter holder: ``proj = Conv2d(in_chans, embed_dim, kernel=stride=patch)``."""

    def __init__(self, img_size, patch_size, in_chans, embed_dim):
        super().__init__()
        self.img_size = (img_size, img_size)
        self.patch_size = (patch_size, patch_size)
        self.grid_size = (img_size // patch_size, img_size // patch_size)
        self.num_patches = self.grid_size[0] * self.grid_size[1]
        self.proj = nn.Conv2d(in_chans, embed_dim, kernel_size=patch_size, stride=patch_size, bias=True)


class _Mlp(nn.Module):
    def __init__(self, dim, hidden):
        super().__init__()
        self.fc1 = nn.Linear(dim, hidden)
        self.fc2 = nn.Linear(hidden, dim)


class _Attention(nn.Module):
    """parameter holder for Attention (reference vision_transformer.py:13-80)"""

    def __init__(self, dim, num_heads, qkv_bias):
        super().__init__()
        assert dim % num_heads == 0, 'dim should be divisible by num_heads'
        self.num_heads = num_heads
        self.head_dim = dim // num_heads
        self.scale = self.head_dim ** -0.5
        self.qkv = nn.Linear(dim, dim * 3, bias=qkv_bias)
        self.proj = nn.Linear(dim, dim)
        self.keep_attn = False


class _CrossAttention(nn.Module):
    """parameter holder for CrossAttention (reference vision_transformer.py:130-200)"""

    def __init__(self, dim, num_heads, qkv_bias):
        super().__init__()
        assert dim % num_heads == 0, 'dim should be divisible by num_heads'
        self.num_heads = num_heads
        self.head_dim = dim // num_heads
        self.scale = self.head_dim ** -0.5
        self.q = nn.Linear(dim, dim, bias=qkv_bias)
        self.kv = nn.Linear(dim, dim * 2, bias=qkv_bias)
        self.proj = nn.Linear(dim, dim)
        self.keep_attn = False


class _Block(nn.Module):
    """parameter holder for Block (reference vision_transformer.py:83-127)"""

    def __init__(self, dim, num_heads, mlp_ratio, qkv_bias, norm_layer):
        super().__init__()
        self.norm1 = norm_layer(dim)
        self.attn = _Attention(dim, num_heads, qkv_bias)
        self.norm2 = norm_layer(dim)
        self.mlp = _Mlp(dim, int(dim * mlp_ratio))


class _CrossBlock(nn.Module):
    """parameter holder for CrossBlock (reference vision_transformer.py:213-272)"""

    def __init__(self, dim, num_heads, mlp_ratio, qkv_bias, norm_layer):
        super().__init__()
        self.norm1 = norm_layer(dim)
        self.attn = _Attention(dim, num_heads, qkv_bias)
        self.norm_cross = norm_layer(dim)
        self.norm_context = norm_layer(dim)
        self.cross_attn = _CrossAttention(dim, num_heads, qkv_bias)
        self.norm2 = norm_layer(dim)
        self.mlp = _Mlp(dim, int(dim * mlp_ratio))


def _init_vit_timm(module):
    """timm 0.9.2 ``init_weights_vit_timm``: Linear -> trunc_normal(std .02), zero bias. It runs inside
    ``VisionTransformer.__init__`` i.e. BEFORE the reference creates ``cross_blocks`` (vision_transformer.py:344-368),
    so cross blocks keep PyTorch's default init -- mirrored here."""
    if isinstance(module, nn.Linear):
        nn.init.trunc_normal_(module.weight, std=.02)
        if module.bias is not None:
            nn.init.zeros_(module.bias)


class VisionTransformerCustom(nn.Module):
    """ViT encoder-decoder pair scorer; drop-in for reference models/vision_transformer.py:275-420."""

    def __init__(
            self,
            img_size=224,
            patch_size=16,
            in_chans=3,
            num_classes=1000,
            global_pool='token',
            embed_dim=768,
            depth=12,
            c_depth=12,
            num_heads=12,
            mlp_ratio=4.,
            qkv_bias=True,
            qk_norm=False,
            init_values=None,
            class_token=True,
            no_embed_class=False,
            pre_norm=False,
            fc_norm=None,
            drop_rate=0.,
            pos_drop_rate=0.,
            patch_drop_rate=0.,
            proj_drop_rate=0.,
            attn_drop_rate=0.,
            drop_path_rate=0.,
            weight_init='',
            embed_layer=None,
            norm_layer=None,
            act_layer=None,
            block_fn=None,
            cross_block_fn=None,
            mlp_layer=None,
            keep_attn=False,
            arch_version='v1',
    ):
        super().__init__()
        # Options build_model() never sets (models/build.py:19-32) are Identity / defaults in the reference at eval;
        # anything else would change the arithmetic of the hot path and is rejected rather than silently ignored.
        unsupported = dict(global_pool=(global_pool, 'token'), qk_norm=(qk_norm, False), init_values=(init_values, None),
                           class_token=(class_token, True), no_embed_class=(no_embed_class, False),
                           pre_norm=(pre_norm, False), fc_norm=(fc_norm, None), weight_init=(weight_init, ''),
                           embed_layer=(embed_layer, None), norm_layer=(norm_layer, None), act_layer=(act_layer, None),
                           block_fn=(block_fn, None), cross_block_fn=(cross_block_fn, None), mlp_layer=(mlp_layer, None))
        for k, (got, want) in unsupported.items():
            if got != want:
                raise NotImplementedError(f'{k}={got!r} is outside the all-pairs scoring path (only {want!r})')
        if isinstance(img_size, (tuple, list)):
            assert img_size[0] == img_size[1], 'square inputs only'
            img_size = img_size[0]
        if isinstance(patch_size, (tuple, list)):
            assert patch_size[0] == patch_size[1], 'square patches only'
            patch_size = patch_size[0]
        assert embed_dim % num_heads == 0, 'dim should be divisible by num_heads'
        norm_layer = partial(nn.LayerNorm, eps=1e-6)

        self.num_classes = num_classes
        self.global_pool = global_pool
        self.num_features = self.embed_dim = embed_dim
        self.num_prefix_tokens = 1
        self.img_size = img_size
        self.patch_size = patch_size
        self.in_chans = in_chans
        self.depth = depth
        self.c_depth = c_depth
        self.num_heads = num_heads
        self.mlp_ratio = mlp_ratio
        self.qkv_bias = qkv_bias
        # dropout-style arguments are accepted for signature parity; they are identity at eval (SURVEY 3.3)
        self.drop_rates = dict(drop=drop_rate, pos=pos_drop_rate, patch=patch_drop_rate, proj=proj_drop_rate,
                               attn=attn_drop_rate, path=drop_path_rate)

        self.patch_embed = _PatchEmbed(img_size, patch_size, in_chans, embed_dim)
        num_patches = self.patch_embed.num_patches
        self.cls_token = nn.Parameter(torch.zeros(1, 1, embed_dim))
        self.pos_embed = nn.Parameter(torch.randn(1, num_patches + 1, embed_dim) * .02)
        self.blocks = nn.Sequential(*[
            _Block(embed_dim, num_heads, mlp_ratio, qkv_bias, norm_layer) for _ in range(depth)])
        self.norm = norm_layer(embed_dim)
        self.head = nn.Linear(embed_dim, num_classes) if num_classes > 0 else nn.Identity()
        # timm init (runs before cross_blocks exist in the reference)
        nn.init.trunc_normal_(self.pos_embed, std=.02)
        nn.init.normal_(self.cls_token, std=1e-6)
        self.apply(_init_vit_timm)
        self.cross_blocks = nn.ModuleList([
            _CrossBlock(embed_dim, num_heads, mlp_ratio, qkv_bias, norm_layer) for _ in range(c_depth)])
        self.keep_attn = keep_attn
        if keep_attn:
            raise NotImplementedError('keep_attn=True (attention-map visualisation) is outside the scoring path')
        self.arch_version = arch_version.lower()

        self._engine = None
        self._engine_device = None
        self._synced_versions = None

    # ------------------------------------------------------------------ engine plumbing
    def _config(self):
        return _lib.Config(self.img_size, self.patch_size, self.in_chans, self.num_classes, self.embed_dim, self.depth,
                           self.c_depth, self.num_heads, float(self.mlp_ratio), int(bool(self.qkv_bias)))

    def _param_versions(self):
        return tuple((p.data_ptr(), p._version) for p in self.parameters())

    def _check_device(self, device):
        if device.type != 'cuda':
            raise _lib.VitedError('vit-ed_b200 runs on CUDA (sm_100a) tensors only; there is no CPU fallback')
        first = next(self.parameters())
        if first.device != device:
            raise _lib.VitedError(f'model parameters are on {first.device}, input is on {device}; call model.cuda()')

    def _ensure_engine(self, device):
        self._check_device(device)
        index = device.index if device.index is not None else torch.cuda.current_device()
        if self._engine is None or self._engine_device != index:
            self._release_engine()
            handle = ctypes.c_void_p()
            cfg = self._config()
            _lib.check(_lib.lib.vited_create(ctypes.byref(cfg), index, ctypes.byref(handle)), 'vited_create')
            self._engine = handle
            self._engine_device = index
            self._synced_versions = None
        versions = self._param_versions()
        if versions != self._synced_versions:
            self._upload_weights()
            self._synced_versions = versions
        return self._engine

    def _upload_weights(self):
        stream = self._stream(torch.device('cuda', self._engine_device))
        sd = self.state_dict()
        n_expected = _lib.lib.vited_num_weights_expected(self._engine)
        expected = [_lib.lib.vited_weight_name(self._engine, i).decode() for i in range(n_expected)]
        missing = [k for k in expected if k not in sd]
        if missing:
            raise _lib.VitedError(f'state_dict lacks keys the engine needs: {missing[:5]}...')
        for name in expected:
            t = sd[name].detach()
            if t.dtype != torch.float32:
                t = t.float()
            t = t.contiguous()
            _lib.check(_lib.lib.vited_load_weight(self._engine, name.encode(), ctypes.c_void_p(t.data_ptr()),
                                                  t.numel(), stream), f'vited_load_weight({name})')

    def _release_engine(self):
        if getattr(self, '_engine', None) is not None:
            _lib.lib.vited_destroy(self._engine)
            self._engine = None

    def __del__(self):
        try:
            self._release_engine()
        except Exception:
            pass

    def set_option(self, option, value):
        """Engine knobs (debug kernels, chunk rows, memory budgets, profiling); see include/vited_b200.h."""
        if self._engine is None:
            self._ensure_engine(next(self.parameters()).device)
        _lib.check(_lib.lib.vited_set_option(self._engine, int(option), int(value)), 'vited_set_option')

    def profile_read(self):
        """dict: per-kernel-class device time / algorithmic flops / bytes since OPT_PROFILE was set (resets)."""
        import json
        if self._engine is None:
            return {}
        return json.loads(_lib.lib.vited_profile_json(
            self._engine, self._stream(torch.device('cuda', self._engine_device))).decode())

    def launch_count(self):
        return int(_lib.lib.vited_launch_count(self._engine)) if self._engine is not None else 0

    @staticmethod
    def _stream(device):
        """The caller's current stream ON THE TENSORS' DEVICE (not on torch's current device, which may be another
        GPU); the C entry points make that device current for their own duration and restore the caller's."""
        return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)

    @staticmethod
    def _prep(t):
        t = t.detach()
        if t.dtype != torch.float32:
            t = t.float()
        return t.contiguous()

    # ------------------------------------------------------------------ reference API
    _ENCODE_PARAMS = ('patch_embed.proj.', 'pos_embed', 'blocks.')
    _DECODE_PARAMS = ('patch_embed.proj.', 'cls_token', 'pos_embed', 'cross_blocks.', 'norm.', 'head.')

    def _mode_params(self, prefixes):
        """(names, parameters) of one forward mode: what the reference's graph of that mode uses."""
        named = [(n, p) for n, p in self.named_parameters() if n.startswith(prefixes)]
        return [n for n, _ in named], [p for _, p in named]

    def _differentiable(self, params, *inputs):
        """A forward runs through torch.autograd (train.encode / train.decode, the training kernels) only when the
        caller is training: grad mode on, the module in training mode, and a parameter of the mode or a floating-point
        input requiring grad. Everything else -- eval(), no_grad, inference_mode, frozen parameters -- runs the scoring
        engine. Train and eval compute the same function here (no dropout, no BatchNorm)."""
        if not (torch.is_grad_enabled() and self.training):
            return False
        return any(p.requires_grad for p in params) or any(t.is_floating_point() and t.requires_grad for t in inputs)

    def forward_first_part(self, x1):
        """[B, C, S, S] -> encoder tokens [B, N_e, D] (reference vision_transformer.py:382-388)."""
        images = x1
        x1 = self._prep(x1)
        self._check_images(x1)
        names, params = self._mode_params(self._ENCODE_PARAMS)
        if self._differentiable(params, images):
            self._check_device(x1.device)
            return train.encode(self, images, names, params)
        return self._encode(x1)

    @torch.no_grad()
    def _encode(self, x1):
        eng = self._ensure_engine(x1.device)
        out = torch.empty((x1.shape[0], self.patch_embed.num_patches, self.embed_dim), dtype=torch.float32,
                          device=x1.device)
        _lib.check(_lib.lib.vited_encode(eng, x1.data_ptr(), x1.shape[0], out.data_ptr(), self._stream(x1.device)),
                   'vited_encode')
        return out

    def forward(self, x, x2=None, forward_first_part=False):
        """Three modes, as reference vision_transformer.py:412-420. In training mode with gradients wanted (see
        ``_differentiable``) each mode is a torch.autograd Function: ``loss.backward()`` reaches the parameters, the
        context tokens and images that require grad. The backward runs at loss scale 1: the 16-bit gradient operands
        carry whatever scale the caller applied (torch.amp.GradScaler), and so does ``p.grad``, as under fp16
        autocast. A 16-bit overflow in the backward shows as +inf in the gradients, where GradScaler looks for it.
        Like fp16 autocast without a scaler, an fp16 build can underflow small gradients; a bf16 build cannot."""
        if forward_first_part:
            return self.forward_first_part(x)
        if x2 is not None:
            tokens, images = x, x2
            x = self._prep(x)
            x2 = self._prep(x2)
            self._check_images(x2)
            n_e = self.patch_embed.num_patches
            if x.dim() != 3 or x.shape[1] != n_e or x.shape[2] != self.embed_dim or x.shape[0] != x2.shape[0]:
                raise ValueError(f'expected context tokens [{x2.shape[0]}, {n_e}, {self.embed_dim}], got {tuple(x.shape)}')
            self._check_device(x2.device)
            if x.device != x2.device:
                raise _lib.VitedError(f'context tokens are on {x.device}, images on {x2.device}')
            names, params = self._mode_params(self._DECODE_PARAMS)
            if self._differentiable(params, tokens, images):
                return train.decode(self, tokens, images, names, params)
            return self._decode(x, x2)
        pairs = x
        x = self._prep(x)
        if x.dim() != 5 or x.shape[1] != 2:
            raise ValueError(f'expected stacked pairs [B, 2, C, S, S], got {tuple(x.shape)}')
        self._check_images(x[:, 0])
        if self._differentiable(list(self.parameters()), pairs):
            self._check_device(x.device)
            first, second = torch.unbind(pairs, 1)                 # as the reference's forward composes the two parts
            enc_names, enc_params = self._mode_params(self._ENCODE_PARAMS)
            dec_names, dec_params = self._mode_params(self._DECODE_PARAMS)
            tokens = train.encode(self, first, enc_names, enc_params)
            return train.decode(self, tokens, second, dec_names, dec_params)
        return self._forward_pairs(x)

    @torch.no_grad()
    def _decode(self, x, x2):
        eng = self._ensure_engine(x2.device)
        out = torch.empty((x2.shape[0], self.num_classes), dtype=torch.float32, device=x2.device)
        _lib.check(_lib.lib.vited_decode(eng, x.data_ptr(), x2.data_ptr(), x2.shape[0], out.data_ptr(),
                                         self._stream(x2.device)), 'vited_decode')
        return out

    @torch.no_grad()
    def _forward_pairs(self, x):
        eng = self._ensure_engine(x.device)
        out = torch.empty((x.shape[0], self.num_classes), dtype=torch.float32, device=x.device)
        _lib.check(_lib.lib.vited_forward_pairs(eng, x.data_ptr(), x.shape[0], out.data_ptr(), self._stream(x.device)),
                   'vited_forward_pairs')
        return out

    def _check_images(self, t):
        want = (self.in_chans, self.img_size, self.img_size)
        if t.dim() != 4 or tuple(t.shape[1:]) != want:
            raise ValueError(f"Input image size ({tuple(t.shape[1:])}) doesn't match model ({want}).")

    # ------------------------------------------------------------------ grid entry (replaces the L3 loops)
    @torch.no_grad()
    def score_grid(self, images, mode, row_begin=0, row_end=None, out=None):
        """All pairs of grid rows [row_begin, row_end) against all N items -> [rows, N, num_classes] fp32.
        Replaces the inner loops of evaluation.py:101-114 / hisfrag.py:189-231 (see grid.py for the callers).

        ``images`` is either the model input [N, in_chans, S, S] (fp32) or the decoded crops [N, S, S, in_chans] as a
        CUDA uint8 tensor: ToTensor + Normalize(.5, .5) then runs inside the patch embedding (C-ABI
        ``vited_score_grid_u8``), bit-identical to scoring the normalised fp32 images, at a quarter of their memory."""
        images, u8 = self._grid_images(images)
        entry, name = ((_lib.lib.vited_score_grid_u8, 'vited_score_grid_u8') if u8 else
                       (_lib.lib.vited_score_grid, 'vited_score_grid'))
        n = images.shape[0]
        row_end = n if row_end is None else row_end
        if not (0 <= row_begin <= row_end <= n):
            raise _lib.VitedError(f'bad row range [{row_begin}, {row_end}) for N={n}')
        eng = self._ensure_engine(images.device)
        if out is None:
            out = torch.zeros((row_end - row_begin, n, self.num_classes), dtype=torch.float32, device=images.device)
        _lib.check(entry(eng, images.data_ptr(), n, int(mode), int(row_begin), int(row_end), out.data_ptr(),
                         self._stream(images.device)), name)
        return out

    def _grid_images(self, images):
        """The two image forms of score_grid / score_pairs -> (contiguous tensor, is_uint8)."""
        if images.dtype == torch.uint8:
            want = (self.img_size, self.img_size, self.in_chans)
            if images.dim() != 4 or tuple(images.shape[1:]) != want or not images.is_cuda:
                raise ValueError(f'uint8 images must be a CUDA tensor [N, {want[0]}, {want[1]}, {want[2]}] (HWC crops), '
                                 f'got {tuple(images.shape)} on {images.device}')
            return images.contiguous(), True
        images = self._prep(images)
        self._check_images(images)
        return images, False

    @torch.no_grad()
    def score_pairs(self, images, pairs, out=None):
        """Logits of a caller-given pair list -> [P, num_classes] fp32, ``out[p]`` = model(tokens(images[a]), images[b])
        for ``pairs[p] = (a, b)``: the (a, b) entry of ``score_grid``. Any order; duplicates, a == b and a > b are
        allowed. Every item the list references is encoded, and its decoder input state built, once per call (C-ABI
        ``vited_score_pairs``), which is what makes this cheaper than ``model(pairs)`` when items repeat.

        ``images`` takes the two forms of ``score_grid``. ``pairs`` is an int32 / int64 [P, 2] tensor on the images'
        device. An index outside [0, N) raises ``VitedError`` naming the pair, before anything is scored."""
        images, u8 = self._grid_images(images)
        if not isinstance(pairs, torch.Tensor) or pairs.dim() != 2 or pairs.shape[1] != 2:
            raise ValueError(f'pairs must be a [P, 2] tensor, got {getattr(pairs, "shape", type(pairs))}')
        if pairs.dtype not in (torch.int32, torch.int64):
            raise ValueError(f'pairs must be int32 or int64, got {pairs.dtype}')
        if pairs.device != images.device:
            raise ValueError(f'pairs are on {pairs.device}, images on {images.device}')
        if pairs.dtype == torch.int64:      # out-of-range values stay out of range
            pairs = pairs.clamp(-2 ** 31, 2 ** 31 - 1)
        pairs = pairs.to(torch.int32).contiguous()
        n, n_pairs = images.shape[0], pairs.shape[0]
        if out is None:
            out = torch.empty((n_pairs, self.num_classes), dtype=torch.float32, device=images.device)
        elif (out.shape != (n_pairs, self.num_classes) or out.dtype != torch.float32 or out.device != images.device
              or not out.is_contiguous()):
            raise ValueError(f'out must be a contiguous fp32 [{n_pairs}, {self.num_classes}] tensor on {images.device}')
        if n_pairs == 0:
            return out
        eng = self._ensure_engine(images.device)
        entry, name = ((_lib.lib.vited_score_pairs_u8, 'vited_score_pairs_u8') if u8 else
                       (_lib.lib.vited_score_pairs, 'vited_score_pairs'))
        _lib.check(entry(eng, images.data_ptr(), n, pairs.data_ptr(), n_pairs, out.data_ptr(),
                         self._stream(images.device)), name)
        return out


def build_model(config, is_pretrain=False):
    """reference models/build.py:15-32 -- only the ``pjs`` branch is on the all-pairs scoring path."""
    model_type = config.MODEL.TYPE
    if model_type == 'pjs':
        return VisionTransformerCustom(
            img_size=config.DATA.IMG_SIZE,
            patch_size=config.MODEL.PJS.PATCH_SIZE,
            in_chans=config.MODEL.PJS.IN_CHANS,
            num_classes=config.MODEL.NUM_CLASSES,
            embed_dim=config.MODEL.PJS.EMBED_DIM,
            depth=config.MODEL.PJS.DEPTH,
            c_depth=config.MODEL.PJS.C_DEPTH,
            num_heads=config.MODEL.PJS.NUM_HEADS,
            mlp_ratio=config.MODEL.PJS.MLP_RATIO,
            qkv_bias=config.MODEL.PJS.QKV_BIAS,
            keep_attn=config.MODEL.PJS.KEEP_ATTN,
            arch_version=config.MODEL.PJS.ARCH_VERSION,
        )
    raise NotImplementedError(f'Unkown model: {model_type} (only MODEL.TYPE == "pjs" is on the scoring path)')
