"""Host side of the Hisfrag training step (SURVEY 8f row 1): pair construction of ``prepare_data`` (hisfrag.py:117-147)
and one optimisation-free training step -- forward with saved activations, BCE-with-logits, backward to every parameter
(hisfrag.py:149-159 + the autograd pass of misc/engine.py:189-257) -- on this repo's kernels.

The reference's training loop is host Python around GPU kernels; so is this one. PyTorch supplies device buffers and
streams only: every arithmetic step is a C-ABI call (include/vited_b200.h, "Hisfrag training step"). All Linear layers
-- forward, dgrad, wgrad -- run on the tcgen05 GEMM (``vited_op_gemm``) with 16-bit operands; LayerNorm, GELU, softmax
attention (forward and backward), residual adds, gathers / scatter-adds and the loss run in fp32 kernels of
csrc/train_ops.cu. Gradients carry a loss scale (default 1024) while they are 16-bit GEMM operands and are unscaled when
accumulated into the fp32 parameter gradients. There is no PyTorch autograd and no CPU path.

``train_iteration`` completes the reference's iteration (misc/engine.py:189-257, misc/utils.py:206-226) on the device:
the same step with overflow detection for the loss-scaled 16-bit gradients (``LossScaler``, GradScaler's rule),
gradient-norm clipping and a fused ``AdamW`` step (csrc/train_optim.cu).

Not built yet (DESIGN.md): tensor-core attention backward (the softmax attention here is a plain fp32 kernel pair),
DDP gradient all-reduce overlap.
"""
import ctypes
import math
import struct

import numpy as np
import torch

from . import _lib


def prepare_pairs(targets, generator=None):
    """(groups [P, 2] int64, labels [P, 1] fp32) of one batch, as HisfragTrainer.prepare_data builds them
    (hisfrag.py:117-147): for every item i the later items j > i of the same writer are positive pairs (i, j), those of
    another writer negative pairs; at most twice as many negatives as positives survive a ``torch.randperm`` draw
    (``generator`` seeds it; None = the global RNG as in the reference); positives first. The decoder then scores
    ``model(tokens[groups[:, 1]], images[groups[:, 0]])`` (:152-159)."""
    t = torch.as_tensor(targets).view(-1).cpu()
    n = t.numel()
    same = t.view(-1, 1) == t.view(1, -1)
    upper = torch.triu(torch.ones(n, n, dtype=torch.bool), diagonal=0)
    pos = torch.nonzero(same & torch.triu(torch.ones(n, n, dtype=torch.bool), diagonal=1))   # row-major = i-major, j ascending
    neg = torch.nonzero(~same & upper)
    keep = min(neg.shape[0], int(2 * pos.shape[0]))
    perm = torch.randperm(neg.shape[0], generator=generator) if generator is not None else torch.randperm(neg.shape[0])
    neg = neg[perm[:keep]]
    labels = torch.cat([torch.ones(pos.shape[0]), torch.zeros(neg.shape[0])]).view(-1, 1)
    return torch.cat([pos, neg], dim=0), labels


# ----------------------------------------------------------------------------------------------------------------
# thin wrappers: torch tensors in, C-ABI calls out
# ----------------------------------------------------------------------------------------------------------------
def _p(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


class _Ops:
    """One object per training step: device, stream, the 16-bit type, the loss scale and the gradient store. With an
    overflow ``flag`` (one int32 on the device) every loss-scaled gradient that is converted to or from 16 bits is
    range-checked into it; without one (``train_step``) nothing is checked and no extra kernel runs. ``grads``
    (name -> zeroed fp32 tensor) makes the step accumulate into caller-owned gradient buffers."""

    def __init__(self, device, loss_scale, flag=None, grads=None):
        self.dev = device
        self.act = _lib.act_dtype()
        self.S = float(loss_scale)
        self.stream = ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)
        self.flag = flag
        self.limit = _lib.range_limit()
        self.grads = dict(grads) if grads is not None else {}
        self.w16, self.w16t = {}, {}
        self.launches = 0
        self.profile = None          # {op name: [events]} when train_step(profile=True): per-kernel-class device time
        self._last = None

    def _chk(self, status, what):
        self.launches += 1
        _lib.check(status, what)
        if self.profile is not None:
            ev = torch.cuda.Event(enable_timing=True)
            ev.record(torch.cuda.current_stream(self.dev))
            self.profile.append((what, self._last, ev))
            self._last = ev

    def profile_begin(self):
        self.profile = []
        self._last = torch.cuda.Event(enable_timing=True)
        self._last.record(torch.cuda.current_stream(self.dev))

    def profile_read(self):
        torch.cuda.synchronize(self.dev)
        out = {}
        for what, a, b in self.profile:
            ms, n = out.get(what, (0.0, 0))
            out[what] = (ms + a.elapsed_time(b), n + 1)
        return {k: {'ms': round(v[0], 3), 'launches': v[1]} for k, v in sorted(out.items(), key=lambda kv: -kv[1][0])}

    def empty(self, *shape, dtype=torch.float32):
        return torch.empty(shape, dtype=dtype, device=self.dev)

    def zeros(self, *shape, dtype=torch.float32):
        return torch.zeros(shape, dtype=dtype, device=self.dev)   # (cudaMemset: plumbing, not arithmetic)

    def range_check(self, x):
        """flag = 1 if the contiguous fp32 / 16-bit buffer x holds a value the 16-bit conversion cannot represent"""
        if self.flag is None:
            return
        assert x.is_contiguous(), x.shape
        self._chk(_lib.lib.vited_train_range_check(_p(x), 1 if x.dtype == torch.float32 else 0, x.numel(), self.limit,
                                                   _p(self.flag), self.stream), 'train_range_check')

    # ---- casts / adds
    def cast(self, x32, scale=1.0):
        out = self.empty(*x32.shape, dtype=self.act)
        self._chk(_lib.lib.vited_train_cast(_p(x32), _p(out), x32.numel(), scale, self.stream), 'train_cast')
        return out

    def to_f32(self, x16, out=None, alpha=1.0, beta=0.0):
        out = self.empty(*x16.shape) if out is None else out
        self._chk(_lib.lib.vited_train_axpby16(_p(x16), _p(out), x16.numel(), alpha, beta, self.stream), 'train_axpby16')
        return out

    def add_(self, y32, x32, alpha=1.0):
        self._chk(_lib.lib.vited_train_axpy32(_p(x32), _p(y32), x32.numel(), alpha, self.stream), 'train_axpy32')
        return y32

    def transpose(self, x, scale=1.0):
        """[R, C] (fp32 or 16-bit) -> 16-bit [C, ceil8(R)], the padding columns zero."""
        r, c = x.shape
        rp = (r + 7) // 8 * 8
        out = self.empty(c, rp, dtype=self.act)
        self._chk(_lib.lib.vited_train_transpose(_p(x), 1 if x.dtype == torch.float32 else 0, c, _p(out), rp, r, c, scale,
                                                 self.stream), 'train_transpose')
        return out

    # ---- GEMM on the tcgen05 kernel: C16[M, N] = A16[M, K] W16[N, K]^T + bias
    def gemm(self, a16, w16, bias32):
        m, k = a16.shape
        n = w16.shape[0]
        assert w16.shape[1] == k and k % 8 == 0 and n % 8 == 0, (a16.shape, w16.shape)
        out = self.empty(m, n, dtype=self.act)
        self._chk(_lib.lib.vited_op_gemm(_p(a16), _p(w16), _p(bias32), _p(out), m, n, k, 0, 0, self.stream), 'op_gemm')
        return out

    # ---- parameters
    def weight16(self, name, w32):
        if name not in self.w16:
            w = w32.reshape(w32.shape[0], -1)
            if w.shape[0] % 8:                                   # the head (num_classes rows): pad the output dim to 8
                pad = self.zeros(8 - w.shape[0] % 8, w.shape[1])
                w = torch.cat([w, pad], dim=0)                   # (concatenation of buffers: plumbing)
            self.w16[name] = self.cast(w.contiguous())
            self.w16t[name] = self.transpose(self.w16[name])     # [K, ceil8(N)] for dgrad
        return self.w16[name], self.w16t[name]

    def grad(self, name, like):
        if name not in self.grads:
            self.grads[name] = torch.zeros_like(like, dtype=torch.float32)
        return self.grads[name]


class _Linear:
    """y = x W^T + b with everything its backward needs (the 16-bit input)."""

    def __init__(self, ops, sd, prefix):
        self.ops, self.prefix = ops, prefix
        self.w32, self.b32 = sd[prefix + '.weight'], sd[prefix + '.bias']
        self.n_out = self.w32.shape[0]
        self.w16, self.w16t = ops.weight16(prefix + '.weight', self.w32)
        self.n_pad = self.w16.shape[0]
        self.bias = self.b32 if self.n_pad == self.n_out else torch.cat([self.b32, ops.zeros(self.n_pad - self.n_out)])
        self.zero_bias_in = ops.zeros(self.w16.shape[1])
        self.x16 = None

    def forward(self, x16):
        self.x16 = x16
        return self.ops.gemm(x16, self.w16, self.bias)           # [R, n_pad] 16-bit

    def backward(self, dy32, need_dx=True):
        """dy32 [R, n_pad] fp32 (loss-scaled). Accumulates dW, db (unscaled); returns dx32 [R, K] (loss-scaled)."""
        ops = self.ops
        r = dy32.shape[0]
        inv = 1.0 / ops.S
        gw = ops.grad(self.prefix + '.weight', self.w32)
        gb = ops.grad(self.prefix + '.bias', self.b32)
        ops.range_check(dy32)                                     # before its 16-bit transpose and cast
        # wgrad: dW[N, K] = dY^T[N, R] X[R, K]  ->  gemm(A = dY^T [N, Rp], W = X^T [K, Rp])
        dyt16 = ops.transpose(dy32)
        xt16 = ops.transpose(self.x16)
        dw16 = ops.gemm(dyt16, xt16, self.zero_bias_in)          # [n_pad, K]
        ops.range_check(dw16)
        ops.to_f32(dw16[:self.n_out], out=gw.view(self.n_out, -1), alpha=inv, beta=1.0)
        if self.n_pad == self.n_out:
            ops._chk(_lib.lib.vited_train_colsum(_p(dy32), _p(gb), r, self.n_out, inv, ops.stream), 'train_colsum')
        else:
            tmp = ops.zeros(self.n_pad)
            ops._chk(_lib.lib.vited_train_colsum(_p(dy32), _p(tmp), r, self.n_pad, inv, ops.stream), 'train_colsum')
            ops.add_(gb, tmp[:self.n_out].contiguous())
        if not need_dx:
            return None
        # dgrad: dX[R, K] = dY[R, N] W[N, K]  ->  gemm(A = dY16 [R, n_pad], W = W^T [K, n_pad])
        dy16 = ops.cast(dy32)
        dx16 = ops.gemm(dy16, self.w16t, self.zero_bias_in)
        ops.range_check(dx16)
        return ops.to_f32(dx16)


class _LayerNorm:
    def __init__(self, ops, sd, prefix):
        self.ops, self.prefix = ops, prefix
        self.w, self.b = sd[prefix + '.weight'], sd[prefix + '.bias']

    def forward(self, x32):
        ops = self.ops
        r, d = x32.shape
        self.x = x32
        self.stats = ops.empty(r, 2)
        h16 = ops.empty(r, d, dtype=ops.act)
        ops._chk(_lib.lib.vited_train_ln_forward(_p(x32), _p(self.w), _p(self.b), _p(h16), _p(self.stats), r, d, 1e-6,
                                                 ops.stream), 'train_ln_forward')
        return h16

    def backward(self, dh32, dx32):
        """dx32 += dLN/dx; accumulates the (unscaled) weight / bias gradients."""
        ops = self.ops
        r, d = dh32.shape
        gw, gb = ops.grad(self.prefix + '.weight', self.w), ops.grad(self.prefix + '.bias', self.b)
        ops._chk(_lib.lib.vited_train_ln_backward(_p(dh32), _p(self.x), _p(self.stats), _p(self.w), _p(dx32), _p(gw), _p(gb), r,
                                                  d, 1.0 / ops.S, ops.stream), 'train_ln_backward')


def _attention(ops, backward, q, k, v, n_seq, heads, hd, tq, tk, o=None, lse=None, d_o=None, dq=None, dk=None, dv=None):
    """q / k / v: 16-bit 2-D views (row stride = their leading dimension). Forward returns (o16 [n_seq * tq, heads * hd],
    lse [n_seq, heads, tq]); the backward pass recomputes the probabilities from lse and takes the forward output o
    (D_i = do_i . o_i)."""
    scale = hd ** -0.5
    if not backward:
        o = ops.empty(n_seq * tq, heads * hd, dtype=ops.act)
    if not backward:
        lse = ops.empty(n_seq, heads, tq)
    dsum = ops.empty(n_seq, heads, tq) if backward else None
    ld = lambda t: t.stride(0) if t is not None else 0
    args = (1 if backward else 0, _p(q), ld(q), _p(k), ld(k), _p(v), ld(v), _p(o), ld(o), _p(lse), _p(d_o), ld(d_o), _p(dsum),
            _p(dq), ld(dq), _p(dk), ld(dk), _p(dv), ld(dv), n_seq, heads, hd, tq, tk, scale)
    if backward and ops.flag is not None:     # dS = P (dP - D) scale is converted to 16 bits inside the kernel
        ops._chk(_lib.lib.vited_train_attention_chk(*args, _p(ops.flag), ops.stream), 'train_attention_chk')
    else:
        ops._chk(_lib.lib.vited_train_attention(*args, ops.stream), 'train_attention')
    return o, lse


class _SelfAttn:
    """x + proj(attention(qkv(norm1(x))))  (Attention.forward, vision_transformer.py:56-80)."""

    def __init__(self, ops, sd, prefix, norm_prefix, heads, n_seq, t):
        self.ops, self.heads, self.n_seq, self.t = ops, heads, n_seq, t
        self.norm = _LayerNorm(ops, sd, norm_prefix)
        self.qkv = _Linear(ops, sd, prefix + '.qkv')
        self.proj = _Linear(ops, sd, prefix + '.proj')

    def forward(self, x32):
        ops = self.ops
        d = x32.shape[1]
        self.hd = d // self.heads
        h16 = self.norm.forward(x32)
        self.qkv16 = self.qkv.forward(h16)                        # [R, 3D]: q | k | v
        q, k, v = self.qkv16[:, :d], self.qkv16[:, d:2 * d], self.qkv16[:, 2 * d:]
        o16, self.lse = _attention(ops, False, q, k, v, self.n_seq, self.heads, self.hd, self.t, self.t)
        y16 = self.proj.forward(o16)
        out = ops.to_f32(y16)
        return ops.add_(out, x32)                                 # residual

    def backward(self, dout32):
        ops = self.ops
        d = dout32.shape[1]
        do32 = self.proj.backward(dout32)
        dqkv = ops.zeros(dout32.shape[0], 3 * d)
        q, k, v = self.qkv16[:, :d], self.qkv16[:, d:2 * d], self.qkv16[:, 2 * d:]
        _attention(ops, True, q, k, v, self.n_seq, self.heads, self.hd, self.t, self.t, o=self.proj.x16, lse=self.lse, d_o=do32,
                   dq=dqkv[:, :d], dk=dqkv[:, d:2 * d], dv=dqkv[:, 2 * d:])
        dh32 = self.qkv.backward(dqkv)
        dx32 = dout32.clone()                                     # residual path (device copy: plumbing)
        self.norm.backward(dh32, dx32)
        return dx32


class _CrossAttn:
    """x + proj(attention(q(norm_cross(x)), kv(norm_context(ctx))))  (CrossAttention.forward, :174-200; CrossBlock :270)."""

    def __init__(self, ops, sd, prefix, heads, n_seq, tq, tk):
        self.ops, self.heads, self.n_seq, self.tq, self.tk = ops, heads, n_seq, tq, tk
        self.norm_x = _LayerNorm(ops, sd, prefix + '.norm_cross')
        self.norm_c = _LayerNorm(ops, sd, prefix + '.norm_context')
        self.q = _Linear(ops, sd, prefix + '.cross_attn.q')
        self.kv = _Linear(ops, sd, prefix + '.cross_attn.kv')
        self.proj = _Linear(ops, sd, prefix + '.cross_attn.proj')

    def forward(self, x32, ctx32):
        ops = self.ops
        d = x32.shape[1]
        self.hd = d // self.heads
        self.q16 = self.q.forward(self.norm_x.forward(x32))
        self.kv16 = self.kv.forward(self.norm_c.forward(ctx32))   # [P * Ne, 2D]: k | v
        o16, self.lse = _attention(ops, False, self.q16, self.kv16[:, :d], self.kv16[:, d:], self.n_seq, self.heads, self.hd,
                                   self.tq, self.tk)
        out = ops.to_f32(self.proj.forward(o16))
        return ops.add_(out, x32)

    def backward(self, dout32, dctx32):
        ops = self.ops
        d = dout32.shape[1]
        do32 = self.proj.backward(dout32)
        dq = ops.zeros(*self.q16.shape)
        dkv = ops.zeros(*self.kv16.shape)
        _attention(ops, True, self.q16, self.kv16[:, :d], self.kv16[:, d:], self.n_seq, self.heads, self.hd, self.tq, self.tk,
                   o=self.proj.x16, lse=self.lse, d_o=do32, dq=dq, dk=dkv[:, :d], dv=dkv[:, d:])
        dx32 = dout32.clone()
        self.norm_x.backward(self.q.backward(dq), dx32)
        self.norm_c.backward(self.kv.backward(dkv), dctx32)       # accumulates into the context gradient
        return dx32


class _Mlp:
    """x + fc2(GELU(fc1(norm2(x))))  (timm Mlp; Block :126, CrossBlock :272)."""

    def __init__(self, ops, sd, prefix, norm_prefix):
        self.ops = ops
        self.norm = _LayerNorm(ops, sd, norm_prefix)
        self.fc1 = _Linear(ops, sd, prefix + '.fc1')
        self.fc2 = _Linear(ops, sd, prefix + '.fc2')

    def forward(self, x32):
        ops = self.ops
        self.z16 = self.fc1.forward(self.norm.forward(x32))
        a16 = ops.empty(*self.z16.shape, dtype=ops.act)
        ops._chk(_lib.lib.vited_train_gelu_forward(_p(self.z16), _p(a16), a16.numel(), ops.stream), 'train_gelu_forward')
        out = ops.to_f32(self.fc2.forward(a16))
        return ops.add_(out, x32)

    def backward(self, dout32):
        ops = self.ops
        da32 = self.fc2.backward(dout32)
        dz32 = ops.empty(*da32.shape)
        ops._chk(_lib.lib.vited_train_gelu_backward(_p(da32), _p(self.z16), _p(dz32), dz32.numel(), ops.stream),
                 'train_gelu_backward')
        dx32 = dout32.clone()
        self.norm.backward(self.fc1.backward(dz32), dx32)
        return dx32


def _gather(ops, src32, idx, n_blocks, rows_per, in_stride, in_off, out, out_stride, out_off, accumulate):
    d = src32.shape[-1]
    ops._chk(_lib.lib.vited_train_gather_rows(_p(src32), _p(idx), _p(out), n_blocks, rows_per, in_stride, in_off, out_stride,
                                              out_off, d, 1 if accumulate else 0, ops.stream), 'train_gather_rows')


def _scatter_add(ops, src32, idx, n_blocks, rows_per, src_stride, src_off, dst, dst_stride, dst_off, alpha=1.0):
    d = src32.shape[-1]
    ops._chk(_lib.lib.vited_train_scatter_add_rows(_p(src32), _p(idx), _p(dst), n_blocks, rows_per, src_stride, src_off,
                                                   dst_stride, dst_off, d, alpha, ops.stream), 'train_scatter_add_rows')


def all_reduce_gradients(model):
    """DistributedDataParallel's gradient averaging (the reference wraps the model in DDP, misc/engine.py:74-77): one
    NCCL all-reduce over a single flat fp32 bucket of every parameter gradient, then 1 / world. No-op without an
    initialised process group. (The overlap of this collective with the backward pass is not built.)"""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return
    params = [p for p in model.parameters() if p.grad is not None]
    flat = torch.cat([p.grad.reshape(-1).float() for p in params])
    dist.all_reduce(flat, op=dist.ReduceOp.SUM)
    flat /= dist.get_world_size()
    off = 0
    for p in params:
        n = p.grad.numel()
        p.grad.copy_(flat[off:off + n].view_as(p.grad))
        off += n


@torch.no_grad()
def train_step(model, samples, targets, generator=None, loss_scale=1024.0, groups=None, labels=None, all_reduce=True,
               profile=False):
    """One training step of HisfragTrainer without the optimiser (hisfrag.py:117-159): the pairs of the batch, the
    forward ``model(tokens[groups[:, 1]], samples[groups[:, 0]])`` with the encoder in the graph, ``BCEWithLogitsLoss``,
    and the backward pass to every parameter. Returns (loss, logits [P, C], groups, labels) and leaves the gradients in
    ``p.grad`` of the model's parameters (fp32), as ``loss.backward()`` would -- averaged over the ranks of an
    initialised process group when ``all_reduce`` (what DistributedDataParallel does). Dropout / stochastic depth are not
    modelled (the reference's DROP_PATH_RATE would have to be 0)."""
    if not (isinstance(samples, torch.Tensor) and samples.is_cuda):
        raise _lib.VitedError('train_step runs on CUDA (sm_100a) tensors only; there is no CPU fallback')
    dev = samples.device
    if groups is None:
        groups, labels = prepare_pairs(targets, generator)
    with torch.cuda.device(dev):
        out = _train_step(model, samples.float().contiguous(), groups, labels, loss_scale, profile)
        if all_reduce:
            all_reduce_gradients(model)
        return out


def _train_step(model, samples, groups, labels, loss_scale, profile=False, flag=None, grads=None):
    dev = samples.device
    ops = _Ops(dev, loss_scale, flag, grads)
    if profile:
        ops.profile_begin()
    sd = {k: v.detach().float().contiguous() for k, v in model.state_dict().items()}
    if next(iter(sd.values())).device != dev:
        raise _lib.VitedError('model parameters and samples are on different devices; call model.cuda()')
    B = samples.shape[0]
    D, heads = model.embed_dim, model.num_heads
    ne = model.patch_embed.num_patches
    nd = ne + 1
    P = groups.shape[0]
    g0 = groups[:, 0].to(device=dev, dtype=torch.int32).contiguous()    # image whose decoder state seeds the pair
    g1 = groups[:, 1].to(device=dev, dtype=torch.int32).contiguous()    # image whose encoder tokens are the context
    zeros_b = torch.zeros(max(B, P), dtype=torch.int32, device=dev)
    y = labels.to(dev).float().contiguous().view(-1)

    # ---------------- forward ----------------
    # patch embedding as an im2col GEMM (timm PatchEmbed; vision_transformer.py:383, :391), shared by both stacks
    kpe = model.in_chans * model.patch_size ** 2
    col16 = ops.empty(B * ne, kpe, dtype=ops.act)
    ops._chk(_lib.lib.vited_op_im2col(_p(samples), _p(col16), B, model.in_chans, model.img_size, model.patch_size, ops.stream),
             'op_im2col')
    patch = _Linear(ops, sd, 'patch_embed.proj')
    tok32 = ops.to_f32(patch.forward(col16))                              # [B * Ne, D]
    pos32 = sd['pos_embed'].view(nd, D)
    cls32 = sd['cls_token'].view(1, D)
    # encoder input: tokens + pos_embed[:, 1:]  (:378-380)
    x = ops.empty(B * ne, D)
    _gather(ops, pos32, zeros_b, B, ne, nd, 1, x, ne, 0, False)
    ops.add_(x, tok32)
    enc = []
    for l in range(model.depth):
        att = _SelfAttn(ops, sd, f'blocks.{l}.attn', f'blocks.{l}.norm1', heads, B, ne)
        mlp = _Mlp(ops, sd, f'blocks.{l}.mlp', f'blocks.{l}.norm2')
        x = mlp.forward(att.forward(x))
        enc.append((att, mlp))
    enc_out = x
    # decoder input (prepare_x2, :390-395) of pair p: cls + pos[0] | tokens of image g0[p] + pos[1:]
    x = ops.empty(P * nd, D)
    _gather(ops, pos32, zeros_b, P, nd, nd, 0, x, nd, 0, False)
    _gather(ops, cls32, zeros_b, P, 1, 1, 0, x, nd, 0, True)
    _gather(ops, tok32, g0, P, ne, ne, 0, x, nd, 1, True)
    ctx = ops.empty(P * ne, D)
    _gather(ops, enc_out, g1, P, ne, ne, 0, ctx, ne, 0, False)
    dec = []
    for l in range(model.c_depth):
        pre = f'cross_blocks.{l}'
        att = _SelfAttn(ops, sd, pre + '.attn', pre + '.norm1', heads, P, nd)
        cross = _CrossAttn(ops, sd, pre, heads, P, nd, ne)
        mlp = _Mlp(ops, sd, pre + '.mlp', pre + '.norm2')
        x = mlp.forward(cross.forward(att.forward(x), ctx))
        dec.append((att, cross, mlp))
    # final norm on the class-token rows, head (:400, :417 -> timm forward_head)
    xc = ops.empty(P, D)
    arange_p = torch.arange(P, dtype=torch.int32, device=dev)
    _gather(ops, x, arange_p, P, 1, nd, 0, xc, 1, 0, False)
    norm = _LayerNorm(ops, sd, 'norm')
    head = _Linear(ops, sd, 'head')
    C = model.num_classes
    logits_pad = ops.to_f32(head.forward(norm.forward(xc)))               # [P, ceil8(C)]
    logits = logits_pad[:, :C].contiguous()
    loss = ops.empty(1)
    dlogits = ops.empty(P * C)
    yy = y if y.numel() == P * C else y.view(P, 1).expand(P, C).contiguous().view(-1)
    ops._chk(_lib.lib.vited_train_bce_logits(_p(logits), _p(yy), P * C, _p(loss), _p(dlogits), ops.S, ops.stream),
             'train_bce_logits')

    # ---------------- backward ----------------
    dl_pad = ops.zeros(P, logits_pad.shape[1])
    dl_pad[:, :C] = dlogits.view(P, C)                                    # (strided device copy: plumbing)
    dxc = ops.zeros(P, D)
    norm.backward(head.backward(dl_pad), dxc)
    dx = ops.zeros(P * nd, D)
    _scatter_add(ops, dxc, arange_p, P, 1, 1, 0, dx, nd, 0)               # only the class-token rows receive gradient
    dctx = ops.zeros(P * ne, D)
    for att, cross, mlp in reversed(dec):
        dx = att.backward(cross.backward(mlp.backward(dx), dctx))
    inv = 1.0 / ops.S
    g_pos = ops.grad('pos_embed', sd['pos_embed']).view(nd, D)
    g_cls = ops.grad('cls_token', sd['cls_token']).view(1, D)
    dtok = ops.zeros(B * ne, D)
    _scatter_add(ops, dx, zeros_b, P, nd, nd, 0, g_pos, nd, 0, alpha=inv)
    _scatter_add(ops, dx, zeros_b, P, 1, nd, 0, g_cls, 1, 0, alpha=inv)
    _scatter_add(ops, dx, g0, P, ne, nd, 1, dtok, ne, 0)
    denc = ops.zeros(B * ne, D)
    _scatter_add(ops, dctx, g1, P, ne, ne, 0, denc, ne, 0)
    dx = denc
    for att, mlp in reversed(enc):
        dx = att.backward(mlp.backward(dx))
    _scatter_add(ops, dx, zeros_b, B, ne, ne, 0, g_pos, nd, 1, alpha=inv)
    ops.add_(dtok, dx)
    patch.backward(dtok, need_dx=False)

    for name, p in model.named_parameters():
        g = ops.grads.get(name)
        p.grad = torch.zeros_like(p) if g is None else g.view_as(p).to(p.dtype)
    model.train_launches = ops.launches
    model.train_profile = ops.profile_read() if profile else None   # time between consecutive calls, by entry point
    return loss[0], logits, groups, labels


# ----------------------------------------------------------------------------------------------------------------
# the optimiser side of the iteration: loss scaling, gradient clipping, AdamW (csrc/train_optim.cu)
# ----------------------------------------------------------------------------------------------------------------
def _f32(x):
    return float(np.float32(x))


class LossScaler:
    """Dynamic loss scale with ``torch.amp.GradScaler``'s update rule and defaults: after a step with an overflow the
    scale is multiplied by ``backoff_factor`` and the step is skipped; after ``growth_interval`` consecutive clean steps
    it is multiplied by ``growth_factor`` (if the result is finite in float32). The scale is a float32 value kept on
    the host, because every training kernel takes it as a scalar. ``state_dict`` uses GradScaler's keys, so either
    class loads the other's state."""

    def __init__(self, init_scale=2. ** 16, growth_factor=2., backoff_factor=.5, growth_interval=2000):
        if not growth_factor > 1.0:
            raise ValueError('growth_factor must be > 1')
        if not backoff_factor < 1.0:
            raise ValueError('backoff_factor must be < 1')
        self.scale = _f32(init_scale)
        self.growth_factor, self.backoff_factor = float(growth_factor), float(backoff_factor)
        self.growth_interval = int(growth_interval)
        self._growth_tracker = 0

    def update(self, found_inf):
        """One step of torch's ``_amp_update_scale_`` (float32 scale, double factors)."""
        if found_inf:
            self.scale = _f32(self.scale * self.backoff_factor)
            self._growth_tracker = 0
            return
        successful = self._growth_tracker + 1
        if successful == self.growth_interval:
            with np.errstate(over='ignore'):
                grown = np.float32(self.scale * self.growth_factor)
            if np.isfinite(grown):
                self.scale = float(grown)
            self._growth_tracker = 0
        else:
            self._growth_tracker = successful

    def state_dict(self):
        return {'scale': self.scale, 'growth_factor': self.growth_factor, 'backoff_factor': self.backoff_factor,
                'growth_interval': self.growth_interval, '_growth_tracker': self._growth_tracker}

    def load_state_dict(self, state_dict):
        if not state_dict:
            raise RuntimeError('The source state dict is empty, possibly because it was saved from a disabled instance.')
        self.scale = _f32(state_dict['scale'])
        self.growth_factor = float(state_dict['growth_factor'])
        self.backoff_factor = float(state_dict['backoff_factor'])
        self.growth_interval = int(state_dict['growth_interval'])
        self._growth_tracker = int(state_dict['_growth_tracker'])


def default_no_decay(name, param):
    """The Swin-style ``set_weight_decay`` rule: 1-D parameters, ``*.bias`` and the model's ``no_weight_decay`` names
    (``pos_embed``, ``cls_token``) get no weight decay."""
    return param.dim() == 1 or name.endswith('.bias') or name in ('pos_embed', 'cls_token')


def _double_bits(x):
    return struct.unpack('<q', struct.pack('<d', float(x)))[0]


class AdamW:
    """``torch.optim.AdamW`` (single-tensor form) for the Hisfrag model, as one fused kernel per step over every
    parameter, with the two parameter groups of the reference's ``build_optimizer`` (misc/optimizer.py:12-46): weight
    decay ``weight_decay`` and 0 for the parameters ``default_no_decay`` selects. That rule is the Swin-style
    ``set_weight_decay`` the reference is described as using; it has not been checked against misc/optimizer.py itself.
    ``no_decay`` (a set of parameter names) replaces it.

    Device state: ``exp_avg`` and ``exp_avg_sq`` in fp32, the gradient buffers ``train_iteration`` accumulates into
    (one flat buffer with a slot for the overflow flag, so the all-reduce is one collective), and the pointer tables of
    the norm and AdamW kernels, uploaded once (rebuilt if the parameters move). ``lr`` is an attribute the caller sets
    before each step (the learning-rate schedule stays with the caller). ``state_dict`` / ``load_state_dict`` use
    torch.optim.AdamW's format, so optimizer state moves between the two in both directions."""

    N_PARTIALS = 148 * 8       # blocks of the gradient-norm kernel: part of what makes the norm bit-reproducible
    _ALIGN = 128               # gradient / moment slots start at 512-byte boundaries, as torch allocations do

    def __init__(self, model, lr, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.05, no_decay=None):
        self.lr, self.betas, self.eps = float(lr), (float(betas[0]), float(betas[1])), float(eps)
        self.weight_decay = float(weight_decay)
        params = dict(model.named_parameters())
        skip = set(no_decay) if no_decay is not None else {n for n, p in params.items() if default_no_decay(n, p)}
        unknown = skip - set(params)
        if unknown:
            raise ValueError(f'no_decay names that are not parameters of the model: {sorted(unknown)[:5]}')
        self.groups = [[n for n in params if n not in skip], [n for n in params if n in skip]]
        self.group_decay = [self.weight_decay, 0.0]
        self.names = self.groups[0] + self.groups[1]     # torch's parameter index order in the state_dict
        self.t = 0
        self.params = params
        self.dev = next(iter(params.values())).device     # the step itself runs in train_iteration, on CUDA only
        offs, total = [], 0
        for n in self.names:
            offs.append(total)
            total += (params[n].numel() + self._ALIGN - 1) // self._ALIGN * self._ALIGN
        z = lambda k: torch.zeros(k, dtype=torch.float32, device=self.dev)
        self._grad_flat, self._m_flat, self._v_flat = z(total + 1), z(total), z(total)   # + 1: the flag's slot
        view = lambda flat, n, o: flat[o:o + params[n].numel()].view(params[n].shape)
        self.grads = {n: view(self._grad_flat, n, o) for n, o in zip(self.names, offs)}
        self.exp_avg = {n: view(self._m_flat, n, o) for n, o in zip(self.names, offs)}
        self.exp_avg_sq = {n: view(self._v_flat, n, o) for n, o in zip(self.names, offs)}
        self._status = torch.zeros(2, dtype=torch.int32, device=self.dev)   # (float sum of squares, int32 overflow flag)
        self._partials = torch.empty(self.N_PARTIALS, dtype=torch.float64, device=self.dev)
        self._ptrs = None
        self._tables(model)

    def _tables(self, model):
        """Validates every (param, grad, exp_avg, exp_avg_sq) and uploads the kernels' tables, unless the parameters
        are where the current tables point."""
        params = dict(model.named_parameters())
        if sorted(params) != sorted(self.names):
            raise ValueError('the model does not have the parameters this optimizer was built for')
        self.params = params
        ptrs = tuple(params[n].data_ptr() for n in self.names)
        if ptrs == self._ptrs:
            return
        norm_rows, adam_rows = [], []
        decay = {n: self.group_decay[g] for g, names in enumerate(self.groups) for n in names}
        for n in self.names:
            p, g, m, v = params[n], self.grads[n], self.exp_avg[n], self.exp_avg_sq[n]
            for what, t in (('param', p), ('grad', g), ('exp_avg', m), ('exp_avg_sq', v)):
                if t.device != self.dev or t.dtype != torch.float32 or not t.is_contiguous() or t.data_ptr() == 0:
                    raise ValueError(f'{n}: {what} must be a contiguous fp32 tensor on {self.dev}')
                if t.shape != p.shape:
                    raise ValueError(f'{n}: {what} shape {tuple(t.shape)} != parameter shape {tuple(p.shape)}')
            norm_rows.append([g.data_ptr(), g.numel()])
            adam_rows.append([p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), p.numel(), _double_bits(decay[n])])
        self._norm_table = torch.tensor(norm_rows, dtype=torch.int64).to(self.dev)
        self._adam_table = torch.tensor(adam_rows, dtype=torch.int64).to(self.dev)
        self._max_numel = max(r[4] for r in adam_rows)
        self._ptrs = ptrs

    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.dev).cuda_stream)

    def _grad_norm(self):
        """sum of squares of every gradient into _status[0] (float bits), a non-finite one sets the flag _status[1]"""
        _lib.check(_lib.lib.vited_train_grad_norm(_p(self._norm_table), len(self.names), _p(self._partials),
                                                  self.N_PARTIALS, _p(self._status), self._stream()),
                   'vited_train_grad_norm')

    def _step(self, clip_coef):
        self.t += 1
        b1, b2 = self.betas
        _lib.check(_lib.lib.vited_train_adamw(_p(self._adam_table), len(self.names), self._max_numel, self.lr, b1, b2,
                                              self.eps, clip_coef, 1 - b1 ** float(self.t), 1 - b2 ** float(self.t),
                                              self._stream()), 'vited_train_adamw')

    def _torch_groups(self, params):
        return [{'params': [params[n] for n in self.groups[0]], 'weight_decay': self.group_decay[0]},
                {'params': [params[n] for n in self.groups[1]], 'weight_decay': self.group_decay[1]}]

    def state_dict(self):
        """torch.optim.AdamW(...).state_dict() of the same groups, hyperparameters, step and moments (copies)."""
        ref = torch.optim.AdamW(self._torch_groups(self.params), lr=self.lr, betas=self.betas, eps=self.eps,
                                weight_decay=self.weight_decay, foreach=False, fused=False)
        sd = ref.state_dict()
        if self.t > 0:
            sd['state'] = {i: {'step': torch.tensor(float(self.t)), 'exp_avg': self.exp_avg[n].clone(),
                               'exp_avg_sq': self.exp_avg_sq[n].clone()} for i, n in enumerate(self.names)}
        return sd

    def load_state_dict(self, state_dict):
        """Loads a state_dict of this class or of torch.optim.AdamW over the same two groups."""
        groups = state_dict['param_groups']
        if [len(g['params']) for g in groups] != [len(self.groups[0]), len(self.groups[1])]:
            raise ValueError('the state_dict does not have the decay / no-decay groups of this optimizer')
        if len({g['lr'] for g in groups}) != 1 or len({tuple(g['betas']) for g in groups}) != 1 \
                or len({g['eps'] for g in groups}) != 1:
            raise ValueError('lr, betas and eps must be the same in both groups')
        if any(g.get('amsgrad') or g.get('maximize') for g in groups):
            raise ValueError('amsgrad / maximize are not supported')
        self.lr, self.betas, self.eps = float(groups[0]['lr']), tuple(float(b) for b in groups[0]['betas']), float(groups[0]['eps'])
        self.group_decay = [float(g['weight_decay']) for g in groups]
        self.weight_decay = self.group_decay[0]
        index = {i: n for g, names in zip(groups, self.groups) for i, n in zip(g['params'], names)}
        state = state_dict['state']
        steps = {float(s['step']) for s in state.values()}
        if len(steps) > 1:
            raise ValueError('all parameters must have taken the same number of steps')
        if state and len(state) != len(self.names):
            raise ValueError('the state_dict has state for only some of the parameters')
        self.t = int(steps.pop()) if steps else 0
        for n in self.names:
            self.exp_avg[n].zero_()
            self.exp_avg_sq[n].zero_()
        for i, s in state.items():
            self.exp_avg[index[int(i)]].copy_(s['exp_avg'])
            self.exp_avg_sq[index[int(i)]].copy_(s['exp_avg_sq'])
        self._ptrs = None        # the weight decays may have changed: rebuild the tables at the next step


def _all_reduce_with_flag(flat, flag):
    """all_reduce_gradients on the optimizer's flat gradient buffer, whose last slot carries the overflow flag: any
    rank's overflow becomes every rank's, in the same SUM collective."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return
    flat[-1:].copy_(flag)                        # (int32 -> fp32 device copy: plumbing)
    dist.all_reduce(flat, op=dist.ReduceOp.SUM)
    flat /= dist.get_world_size()
    flag.copy_(flat[-1:] > 0)


@torch.no_grad()
def train_iteration(model, samples, targets, optimizer, scaler, clip_grad=5.0, generator=None, groups=None, labels=None,
                    all_reduce=True):
    """One iteration of the reference's training loop (misc/engine.py:189-257): ``train_step`` at the loss scale
    ``scaler.scale`` with every 16-bit conversion of a loss-scaled gradient range-checked on the device, the gradient
    all-reduce (the overflow flag travels in the same bucket), ``clip_grad_norm_(params, clip_grad)`` and an
    ``optimizer`` (``AdamW``) step -- or, when any rank's gradient overflowed, no step and a smaller scale, as
    ``GradScaler`` does. One 8-byte device-to-host read per call (GradScaler.step synchronises once too).

    Returns (loss, logits, groups, labels, grad_norm, skipped). ``grad_norm`` is the total norm clip_grad_norm_ returns
    (a float; inf for a skipped step). ``p.grad`` holds the unclipped averaged gradient afterwards; on a skipped step
    the parameters, the moments and the step count are untouched."""
    if not (isinstance(samples, torch.Tensor) and samples.is_cuda):
        raise _lib.VitedError('train_iteration runs on CUDA (sm_100a) tensors only; there is no CPU fallback')
    dev = samples.device
    if groups is None:
        groups, labels = prepare_pairs(targets, generator)
    with torch.cuda.device(dev):
        optimizer._tables(model)
        status = optimizer._status
        status.zero_()
        optimizer._grad_flat.zero_()
        flag = status[1:]
        loss, logits, groups, labels = _train_step(model, samples.float().contiguous(), groups, labels, scaler.scale,
                                                   flag=flag, grads=optimizer.grads)
        if all_reduce:
            _all_reduce_with_flag(optimizer._grad_flat, flag)
        optimizer._grad_norm()
        host = status.cpu()
        found_inf = bool(host[1])
        if found_inf:
            scaler.update(True)
            model.train_launches += 2
            return loss, logits, groups, labels, math.inf, True
        norm = np.float32(math.sqrt(float(host[:1].view(torch.float32))))
        clip_coef = min(np.float32(1.0), np.float32(clip_grad) / (norm + np.float32(1e-6)))
        optimizer._step(float(clip_coef))
        scaler.update(False)
        model.train_launches += 3
        # the kernel wrote the parameters through raw pointers: bump their versions so that the scoring engine, which
        # re-uploads its packed weights when a parameter's version changes, does not keep the old ones
        torch.autograd.graph.increment_version(list(model.parameters()))
        return loss, logits, groups, labels, float(norm), False
