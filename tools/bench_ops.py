"""Times each kernel of the path in isolation with CUDA events (GPU box only). Prints one JSON line per op with the
achieved TFLOP/s or GB/s against MEASURED_PEAKS.json. Used to fill profiles/ and DESIGN.md, not a test."""
import ctypes
import json
import math
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from vited_b200 import _lib as L  # noqa: E402


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return d['hbm_gbs'], d['bf16_tflops'], 'measured'
    return 6650.0, 1590.0, 'fallback'


def timeit(fn, iters=20, warmup=3, flush=None):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        if flush is not None:
            flush.zero_()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        fn()
        e.record()
        torch.cuda.synchronize()
        ts.append(s.elapsed_time(e))
    ts.sort()
    return ts[len(ts) // 2]


def main():
    hbm, tf, src = peaks()
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device='cuda')
    st = None
    M = 4032 * 65
    D = 384
    out = []
    sections = os.environ.get('OPS', 'all').split(',')      # OPS=gemm,fused,attn,ln (default: all)
    want = lambda name: 'all' in sections or name in sections  # noqa: E731
    if want('gemm'):
        for name, N, K, act in (('qkv', 1152, 384, 0), ('proj', 384, 384, 0), ('fc1_gelu', 1536, 384, 1),
                                ('fc2', 384, 1536, 0), ('kv', 768, 384, 0)):
            A = torch.randn(M, K, device='cuda').to(L.act_dtype())
            W = (torch.randn(N, K, device='cuda') / math.sqrt(K)).to(L.act_dtype())
            b = torch.randn(N, device='cuda')
            C = torch.empty(M, N, dtype=L.act_dtype(), device='cuda')
            ms = timeit(lambda: L.check(L.lib.vited_op_gemm(A.data_ptr(), W.data_ptr(), b.data_ptr(), C.data_ptr(), M, N, K,
                                                              act, 0, st), 'gemm'), flush=flush)
            fl = 2.0 * M * N * K
            by = 2.0 * (M * K + N * K + M * N)
            out.append(dict(op=f'gemm_{name}', M=M, N=N, K=K, ms=ms, tflops=fl / ms / 1e9, tflops_frac=fl / ms / 1e9 / tf,
                            gbs=by / ms / 1e6, gbs_frac=by / ms / 1e6 / hbm, bn=os.environ.get('VITED_GEMM_BN', 'auto')))
            ms = timeit(lambda: torch.matmul(A, W.t(), out=C), flush=flush)
            out.append(dict(op=f'cublas_{name}', M=M, N=N, K=K, ms=ms, tflops=2.0 * M * N * K / ms / 1e9))
    if want('fused'):
        # the two full-row kernels; the 16-epilogue-warp form only exists in -DVITED_EXPERIMENTAL builds (VITED_EPI_WARPS is
        # read at every launch)
        epis = ('8', '16') if 'experimental' in os.environ.get('VITED_LIB', '') else ('8',)
        for epi, name, K in [(e, n, k) for e in epis for n, k in (('proj', 384), ('fc2', 1536))]:
            os.environ['VITED_EPI_WARPS'] = epi
            A = torch.randn(M, K, device='cuda').to(L.act_dtype())
            W = (torch.randn(384, K, device='cuda') / math.sqrt(K)).to(L.act_dtype())
            b = torch.randn(384, device='cuda')
            xx = torch.randn(M, 384, device='cuda')
            lw = torch.ones(384, device='cuda'); lb = torch.zeros(384, device='cuda')
            hh = torch.empty(M, 384, dtype=L.act_dtype(), device='cuda')
            ms = timeit(lambda: L.check(L.lib.vited_op_gemm_resid_ln(A.data_ptr(), W.data_ptr(), b.data_ptr(), xx.data_ptr(), lw.data_ptr(),
                                                                      lb.data_ptr(), hh.data_ptr(), M, 384, K, 1e-6, st), 'gemm_ln'), flush=flush)
            fl = 2.0 * M * 384 * K
            by = M * K * 2 + 384 * K * 2 + M * 384 * (4 + 4 + 2)
            out.append(dict(op=f'gemm_ln_{name}' + ('_epi16' if epi == '16' else ''), M=M, N=384, K=K, ms=ms, tflops=fl / ms / 1e9,
                            gbs=by / ms / 1e6, gbs_frac=by / ms / 1e6 / hbm))
            del A, W, xx, hh
        # fused MLP sub-block + residual + LayerNorm (fc1 -> GELU -> fc2, hidden activations never written)
        hin = torch.randn(M, 384, device='cuda').to(L.act_dtype())
        W1 = (torch.randn(1536, 384, device='cuda') / math.sqrt(384)).to(L.act_dtype())
        W2 = (torch.randn(384, 1536, device='cuda') / math.sqrt(1536)).to(L.act_dtype())
        b1 = torch.randn(1536, device='cuda'); b2 = torch.randn(384, device='cuda')
        xx = torch.randn(M, 384, device='cuda')
        lw = torch.ones(384, device='cuda'); lb = torch.zeros(384, device='cuda')
        hh = torch.empty(M, 384, dtype=L.act_dtype(), device='cuda')
        for epi in epis:
            os.environ['VITED_EPI_WARPS'] = epi
            ms = timeit(lambda: L.check(L.lib.vited_op_mlp_resid_ln(hin.data_ptr(), W1.data_ptr(), b1.data_ptr(), W2.data_ptr(), b2.data_ptr(),
                                                                     xx.data_ptr(), lw.data_ptr(), lb.data_ptr(), hh.data_ptr(), M, 384, 1536,
                                                                     1e-6, st), 'mlp_ln'), flush=flush)
            fl = 4.0 * M * 384 * 1536
            by = M * 384 * (2 + 4 + 4 + 2) + 4 * 384 * 1536
            out.append(dict(op='mlp_ln' + ('_epi16' if epi == '16' else ''), M=M, D=384, hidden=1536, ms=ms, tflops=fl / ms / 1e9,
                            tflops_frac=fl / ms / 1e9 / tf, gbs=by / ms / 1e6, gbs_frac=by / ms / 1e6 / hbm))
        os.environ.pop('VITED_EPI_WARPS', None)
        del hin, xx, hh
        # the decoder's cross projection + residual + norm2 + MLP sub-block in one launch, against the gemm_ln + mlp_ln
        # pair it replaces, at the engine's chunk shape (524,288 rows)
        Mc = 524288
        o = torch.randn(Mc, 384, device='cuda').to(L.act_dtype())
        Wp = (torch.randn(384, 384, device='cuda') / math.sqrt(384)).to(L.act_dtype())
        bp = torch.randn(384, device='cuda')
        xx = torch.randn(Mc, 384, device='cuda')
        hh = torch.empty(Mc, 384, dtype=L.act_dtype(), device='cuda')

        def pair():
            L.check(L.lib.vited_op_gemm_resid_ln(o.data_ptr(), Wp.data_ptr(), bp.data_ptr(), xx.data_ptr(), lw.data_ptr(),
                                                 lb.data_ptr(), hh.data_ptr(), Mc, 384, 384, 1e-6, st), 'gemm_ln')
            L.check(L.lib.vited_op_mlp_resid_ln(hh.data_ptr(), W1.data_ptr(), b1.data_ptr(), W2.data_ptr(), b2.data_ptr(),
                                                xx.data_ptr(), lw.data_ptr(), lb.data_ptr(), hh.data_ptr(), Mc, 384, 1536, 1e-6,
                                                st), 'mlp_ln')

        def fused():
            L.check(L.lib.vited_op_cproj_mlp_resid_ln(o.data_ptr(), Wp.data_ptr(), bp.data_ptr(), xx.data_ptr(), lw.data_ptr(),
                                                      lb.data_ptr(), W1.data_ptr(), b1.data_ptr(), W2.data_ptr(), b2.data_ptr(),
                                                      lw.data_ptr(), lb.data_ptr(), hh.data_ptr(), Mc, 384, 1536, 1e-6, st),
                    'mlp_ln_cproj')

        fl = 2.0 * Mc * 384 * 384 + 4.0 * Mc * 384 * 1536
        for name, fn, per_row in (('gemm_ln_cproj+mlp_ln', pair, 2 * 4608), ('mlp_ln_cproj', fused, 4608)):
            ms = timeit(fn, flush=flush)
            by = Mc * per_row + 2 * 384 * 384 + 4 * 384 * 1536
            out.append(dict(op=name, M=Mc, D=384, hidden=1536, ms=ms, tflops=fl / ms / 1e9, tflops_frac=fl / ms / 1e9 / tf,
                            gbs=by / ms / 1e6, gbs_frac=by / ms / 1e6 / hbm))
        del o, xx, hh
    if want('ln'):
        x = torch.randn(M, D, device='cuda')
        delta = torch.randn(M, D, device='cuda').to(L.act_dtype())
        w = torch.ones(D, device='cuda'); bb = torch.zeros(D, device='cuda')
        h = torch.empty(M, D, dtype=L.act_dtype(), device='cuda')
        ms = timeit(lambda: L.check(L.lib.vited_op_resid_ln(x.data_ptr(), delta.data_ptr(), w.data_ptr(), bb.data_ptr(), h.data_ptr(),
                                                             4032, 64, 1, D, 1e-6, st), 'ln'), flush=flush)
        by = M * D * (4 + 2 + 4 + 2)
        out.append(dict(op='resid_ln', rows=M, ms=ms, gbs=by / ms / 1e6, gbs_frac=by / ms / 1e6 / hbm))
    if want('attn'):
        # attention (puzzle): self and cross. impl0 = tcgen05, impl2 = mma.sync; impl0_pair = two units per tile
        # (attention_pair.cu, experimental builds only, VITED_P64_PAIR=1 is read at every launch)
        P, H, hd, Np = 4032, 12, 32, 64
        qkv = torch.randn(M, 3 * D, device='cuda').to(L.act_dtype())
        o = torch.empty(M, D, dtype=L.act_dtype(), device='cuda')
        variants = ((0, '0', 'impl0'), (2, '0', 'impl2'))
        if 'experimental' in os.environ.get('VITED_LIB', ''):
            variants += ((0, '1', 'impl0_pair'),)
        for impl, pair, tag in variants:
            os.environ['VITED_P64_PAIR'] = pair
            ms = timeit(lambda: L.check(L.lib.vited_op_attention(qkv.data_ptr(), 3 * D, qkv.data_ptr() + 2 * D, 3 * D, qkv.data_ptr() + 4 * D,
                                                                  3 * D, o.data_ptr(), D, P, H, hd, Np, 1, Np, 1, P, None, hd ** -0.5, impl, st),
                                        'attn'), flush=flush)
            fl = 4.0 * P * H * 65 * 65 * hd
            by = M * D * 2 * 4
            out.append(dict(op=f'attn_self_{tag}', ms=ms, tflops=fl / ms / 1e9, gbs=by / ms / 1e6, gbs_frac=by / ms / 1e6 / hbm))
        kv = torch.randn(540 * Np, 2 * D, device='cuda').to(L.act_dtype())
        q = torch.randn(M, D, device='cuda').to(L.act_dtype())
        idx = (torch.arange(P, device='cuda') // 539).int()
        for impl, pair, tag in variants:
            os.environ['VITED_P64_PAIR'] = pair
            ms = timeit(lambda: L.check(L.lib.vited_op_attention(q.data_ptr(), D, kv.data_ptr(), 2 * D, kv.data_ptr() + 2 * D, 2 * D, o.data_ptr(), D,
                                                                  P, H, hd, Np, 1, Np, 0, 540, idx.data_ptr(), hd ** -0.5, impl, st), 'attn'), flush=flush)
            out.append(dict(op=f'attn_cross_{tag}', ms=ms, tflops=4.0 * P * H * 65 * 64 * hd / ms / 1e9, gbs=M * D * 2 * 2 / ms / 1e6))
        os.environ.pop('VITED_P64_PAIR', None)
    for r in out:
        r['peaks'] = src
        print(json.dumps(r))


if __name__ == '__main__':
    main()
