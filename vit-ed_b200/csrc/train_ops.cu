// Kernels of the Hisfrag training step (SURVEY 8f row 1; reference hisfrag.py:117-159, misc/engine.py:189-257): the pieces
// around the tcgen05 GEMM that a forward-with-saved-activations and a backward pass need. The Linear layers -- forward,
// dgrad (dX = dY W) and wgrad (dW = dY^T X) -- all run on gemm_act (gemm_tc.cu) with 16-bit operands: dgrad takes the
// transposed weight as its "weight" operand, wgrad the transposed gradient and the transposed input (both produced by
// the transpose kernels below, padded to a multiple of 8 rows for the TMA strides). Everything elementwise runs in fp32
// on fp32 buffers: LayerNorm forward / backward, GELU forward / backward (exact erf, as timm's Mlp), softmax attention
// forward / backward (probabilities recomputed in the backward pass, nothing quadratic is stored), bias gradients,
// row gather / scatter-add (pairs <-> items), BCE-with-logits. Gradients carry a loss scale so that 16-bit GEMM operands
// do not underflow; parameter gradients are unscaled when they are accumulated (alpha arguments).
// Plain row-major layouts here ([rows, cols], sequences as consecutive token rows, class token first): the split token
// layout of the scoring path is an inference-side optimisation.
#include "kernels.h"
#include <cstdlib>

namespace vited {

namespace {

constexpr int kThreads = 256;
inline int blocks_for(size_t n, int per_block = kThreads, int cap = 148 * 16) {
  size_t b = (n + per_block - 1) / per_block;
  if (b > (size_t)cap) b = cap;
  return b < 1 ? 1 : (int)b;
}

// ---------------------------------------------------------------------------------------------------------------
// casts / transposes / axpy
// ---------------------------------------------------------------------------------------------------------------
__global__ void cast_scale_kernel(const float* __restrict__ in, act_t* __restrict__ out, size_t n, float scale) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    out[i] = f2act(in[i] * scale);
}
// y = alpha * x16 + beta * y
__global__ void act_axpby_kernel(const act_t* __restrict__ x, float* __restrict__ y, size_t n, float alpha, float beta) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    y[i] = alpha * act2f(x[i]) + (beta == 0.f ? 0.f : beta * y[i]);
}
// y += alpha * x (fp32)
__global__ void f32_axpy_kernel(const float* __restrict__ x, float* __restrict__ y, size_t n, float alpha) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    y[i] += alpha * x[i];
}
// out[c, r] = scale * in[r, c] for r < R, zero for R <= r < ld_out (32 x 32 tiles through shared memory)
template <typename TIn>
__global__ void transpose_kernel(const TIn* __restrict__ in, int ld_in, act_t* __restrict__ out, int ld_out, int R, int C,
                                 float scale) {
  __shared__ float tile[32][33];
  const int r0 = blockIdx.y * 32, c0 = blockIdx.x * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int r = r0 + i, c = c0 + threadIdx.x;
    float v = 0.f;
    if (r < R && c < C) {
      if constexpr (sizeof(TIn) == 4) v = (float)in[(size_t)r * ld_in + c];
      else v = act2f(in[(size_t)r * ld_in + c]);
    }
    tile[i][threadIdx.x] = v * scale;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i, r = r0 + threadIdx.x;
    if (c < C && r < ld_out) out[(size_t)c * ld_out + r] = f2act(tile[threadIdx.x][i]);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// LayerNorm (eps 1e-6, one warp per row)
// ---------------------------------------------------------------------------------------------------------------
__global__ void ln_fwd_kernel(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ b,
                              act_t* __restrict__ h, float* __restrict__ stats, int R, int D, float eps) {
  const int lane = threadIdx.x & 31;
  const int warps = (gridDim.x * blockDim.x) >> 5;
  for (int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < R; r += warps) {
    const float* xr = x + (size_t)r * D;
    float s = 0.f;
    for (int d = lane; d < D; d += 32) s += xr[d];
    const float mean = warp_sum(s) / D;
    float ss = 0.f;
    for (int d = lane; d < D; d += 32) { const float t = xr[d] - mean; ss += t * t; }
    const float rstd = rsqrtf(warp_sum(ss) / D + eps);
    for (int d = lane; d < D; d += 32) h[(size_t)r * D + d] = f2act((xr[d] - mean) * rstd * w[d] + b[d]);
    if (lane == 0) { stats[2 * r] = mean; stats[2 * r + 1] = rstd; }
  }
}
// dx += rstd * (g - mean(g) - xhat * mean(g * xhat)), g = dh * w;  dw += alpha * sum_r dh * xhat;  db += alpha * sum_r dh
__global__ void ln_bwd_kernel(const float* __restrict__ dh, const float* __restrict__ x, const float* __restrict__ stats,
                              const float* __restrict__ w, float* __restrict__ dx, float* __restrict__ dw,
                              float* __restrict__ db, int R, int D, float alpha) {
  extern __shared__ float sacc[];   // [2][D] per-block partial sums of dw / db
  for (int d = threadIdx.x; d < 2 * D; d += blockDim.x) sacc[d] = 0.f;
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int warps = (gridDim.x * blockDim.x) >> 5;
  for (int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < R; r += warps) {
    const float mean = stats[2 * r], rstd = stats[2 * r + 1];
    const float* xr = x + (size_t)r * D;
    const float* gr = dh + (size_t)r * D;
    float s1 = 0.f, s2 = 0.f;
    for (int d = lane; d < D; d += 32) {
      const float xh = (xr[d] - mean) * rstd, g = gr[d] * w[d];
      s1 += g;
      s2 += g * xh;
      atomicAdd(&sacc[d], gr[d] * xh);
      atomicAdd(&sacc[D + d], gr[d]);
    }
    s1 = warp_sum(s1) / D;
    s2 = warp_sum(s2) / D;
    for (int d = lane; d < D; d += 32) {
      const float xh = (xr[d] - mean) * rstd, g = gr[d] * w[d];
      dx[(size_t)r * D + d] += rstd * (g - s1 - xh * s2);
    }
  }
  __syncthreads();
  for (int d = threadIdx.x; d < D; d += blockDim.x) {
    atomicAdd(&dw[d], alpha * sacc[d]);
    atomicAdd(&db[d], alpha * sacc[D + d]);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// GELU (exact erf, timm Mlp act_layer = nn.GELU)
// ---------------------------------------------------------------------------------------------------------------
__global__ void gelu_fwd_kernel(const act_t* __restrict__ z, act_t* __restrict__ a, size_t n) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    a[i] = f2act(gelu_erf(act2f(z[i])));
}
// dz = da * (Phi(z) + z * phi(z))
__global__ void gelu_bwd_kernel(const float* __restrict__ da, const act_t* __restrict__ z, float* __restrict__ dz, size_t n) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const float v = act2f(z[i]);
    const float cdf = 0.5f * (1.0f + erff(v * 0.70710678118654752440f));
    const float pdf = 0.39894228040143267794f * expf(-0.5f * v * v);
    dz[i] = da[i] * (cdf + v * pdf);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// bias gradient: db[c] += alpha * sum_r dy[r, c]
// ---------------------------------------------------------------------------------------------------------------
// block (32, 8): thread (tx, ty) sums 4 adjacent columns over rows ty, ty + 8 * gridDim.y, ... (float4 loads, four
// rows in flight), the 8 partial sums of a column group are combined in shared memory, one atomicAdd per column
__global__ void __launch_bounds__(256) colsum_kernel(const float* __restrict__ dy, float* __restrict__ db, int R, int N,
                                                     float alpha) {
  __shared__ float4 part[8][32];
  const int c4 = (blockIdx.x * 32 + threadIdx.x) * 4;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  if (c4 < N) {
    const int step = 8 * gridDim.y;
    int r = blockIdx.y * 8 + threadIdx.y;
    for (; r + 3 * step < R; r += 4 * step) {
      const float4 a = *reinterpret_cast<const float4*>(dy + (size_t)r * N + c4);
      const float4 b = *reinterpret_cast<const float4*>(dy + (size_t)(r + step) * N + c4);
      const float4 c = *reinterpret_cast<const float4*>(dy + (size_t)(r + 2 * step) * N + c4);
      const float4 d = *reinterpret_cast<const float4*>(dy + (size_t)(r + 3 * step) * N + c4);
      acc.x += (a.x + b.x) + (c.x + d.x); acc.y += (a.y + b.y) + (c.y + d.y);
      acc.z += (a.z + b.z) + (c.z + d.z); acc.w += (a.w + b.w) + (c.w + d.w);
    }
    for (; r < R; r += step) {
      const float4 a = *reinterpret_cast<const float4*>(dy + (size_t)r * N + c4);
      acc.x += a.x; acc.y += a.y; acc.z += a.z; acc.w += a.w;
    }
  }
  part[threadIdx.y][threadIdx.x] = acc;
  __syncthreads();
  if (threadIdx.y == 0 && c4 < N) {
    for (int t = 1; t < 8; ++t) {
      const float4 p = part[t][threadIdx.x];
      acc.x += p.x; acc.y += p.y; acc.z += p.z; acc.w += p.w;
    }
    atomicAdd(&db[c4 + 0], alpha * acc.x);
    atomicAdd(&db[c4 + 1], alpha * acc.y);
    atomicAdd(&db[c4 + 2], alpha * acc.z);
    atomicAdd(&db[c4 + 3], alpha * acc.w);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// row gather / scatter-add: out[i, :] = in[idx[i] * rows_per + t, :] for blocks of rows_per consecutive rows
// ---------------------------------------------------------------------------------------------------------------
__global__ void gather_rows_kernel(const float* __restrict__ in, const int* __restrict__ idx, float* __restrict__ out,
                                   int n_out_blocks, int rows_per, int in_block_stride, int in_row_off, int out_block_stride,
                                   int out_row_off, int D, int accumulate) {
  const size_t total = (size_t)n_out_blocks * rows_per * D;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int d = (int)(i % D);
    const size_t row = i / D;
    const int t = (int)(row % rows_per), blk = (int)(row / rows_per);
    float* dst = out + ((size_t)blk * out_block_stride + out_row_off + t) * D + d;
    const float val = in[((size_t)idx[blk] * in_block_stride + in_row_off + t) * D + d];
    *dst = accumulate ? *dst + val : val;
  }
}
__global__ void scatter_add_rows_kernel(const float* __restrict__ src, const int* __restrict__ idx, float* __restrict__ dst,
                                        int n_src_blocks, int rows_per, int src_block_stride, int src_row_off,
                                        int dst_block_stride, int dst_row_off, int D, float alpha) {
  const size_t total = (size_t)n_src_blocks * rows_per * D;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int d = (int)(i % D);
    const size_t row = i / D;
    const int t = (int)(row % rows_per), blk = (int)(row / rows_per);
    atomicAdd(&dst[((size_t)idx[blk] * dst_block_stride + dst_row_off + t) * D + d],
              alpha * src[((size_t)blk * src_block_stride + src_row_off + t) * D + d]);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// col2im: the inverse permutation of im2col_kernel (rowops.cu) for Conv2d(kernel = stride = p). Patches do not
// overlap, so every image element is one column of one patch row and is written once (no atomics). Four consecutive
// px per thread (p % 4 == 0): a 16-byte load from dcol and a 16-byte store into the image row.
// ---------------------------------------------------------------------------------------------------------------
__global__ void col2im_kernel(const float* __restrict__ dcol, float* __restrict__ dimg, int B, int C, int S, int p) {
  const int G = S / p;
  const int K = C * p * p;
  const int segs_per_row = K / 4;
  const size_t total = (size_t)B * G * G * segs_per_row;
  for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const int seg = (int)(idx % segs_per_row);
    const size_t row = idx / segs_per_row;
    const int col = seg * 4;
    const int c = col / (p * p);
    const int py = (col / p) % p;
    const int px = col % p;
    const int t = (int)(row % (G * G));
    const size_t b = row / (G * G);
    const int gy = t / G, gx = t % G;
    const float4 v = *reinterpret_cast<const float4*>(dcol + row * K + col);
    *reinterpret_cast<float4*>(dimg + ((b * C + c) * S + (gy * p + py)) * S + gx * p + px) = v;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// softmax attention, plain layout: q row (s, i) at q[(s * Tq + i) * q_ld + h * hd ...], k / v row (s, j) likewise.
// Three kernels, one warp per row, no atomics and nothing quadratic stored:
//   forward      (per query row i): p = softmax(q_i K^T * scale), o_i = p V, lse_i = log sum exp
//   backward dQ  (per query row i): p recomputed from lse, dP_j = do_i . v_j, D_i = sum_j p_j dP_j (stored),
//                                   dS_j = p_j (dP_j - D_i) * scale, dq_i += dS K
//   backward dKV (per key row j):   the same p_ij / dS_ij for all i, dk_j += dS^T Q, dv_j += P^T dO
// A CTA handles kRowsPerCta consecutive rows of one (sequence, head), its four warps taking rows in turn.
// ---------------------------------------------------------------------------------------------------------------
constexpr int kAttnWarps = 4;
constexpr int kRowsPerCta = 16;

__device__ __forceinline__ float dot_row16(const act_t* __restrict__ a, const act_t* __restrict__ b, int hd) {
  float acc = 0.f;
  for (int d = 0; d < hd; d += 8) {
    const uint4 ua = *reinterpret_cast<const uint4*>(a + d), ub = *reinterpret_cast<const uint4*>(b + d);
    const float2 a0 = unpack_act(ua.x), a1 = unpack_act(ua.y), a2 = unpack_act(ua.z), a3 = unpack_act(ua.w);
    const float2 b0 = unpack_act(ub.x), b1 = unpack_act(ub.y), b2 = unpack_act(ub.z), b3 = unpack_act(ub.w);
    acc += a0.x * b0.x + a0.y * b0.y + a1.x * b1.x + a1.y * b1.y + a2.x * b2.x + a2.y * b2.y + a3.x * b3.x + a3.y * b3.y;
  }
  return acc;
}
__device__ __forceinline__ float dot_row_f32_16(const float* __restrict__ a, const act_t* __restrict__ b, int hd) {
  float acc = 0.f;
  for (int d = 0; d < hd; d += 8) {
    const float4 x0 = *reinterpret_cast<const float4*>(a + d), x1 = *reinterpret_cast<const float4*>(a + d + 4);
    const uint4 ub = *reinterpret_cast<const uint4*>(b + d);
    const float2 b0 = unpack_act(ub.x), b1 = unpack_act(ub.y), b2 = unpack_act(ub.z), b3 = unpack_act(ub.w);
    acc += x0.x * b0.x + x0.y * b0.y + x0.z * b1.x + x0.w * b1.y + x1.x * b2.x + x1.y * b2.y + x1.z * b3.x + x1.w * b3.y;
  }
  return acc;
}

__global__ void __launch_bounds__(32 * kAttnWarps)
attn_fwd_kernel(const act_t* __restrict__ q, int q_ld, const act_t* __restrict__ k, int k_ld, const act_t* __restrict__ v,
                int v_ld, act_t* __restrict__ o, int o_ld, float* __restrict__ lse, int H, int hd, int Tq, int Tk,
                float scale) {
  extern __shared__ float smem_p[];            // [kAttnWarps][Tk]
  const int blocks_per = (Tq + kRowsPerCta - 1) / kRowsPerCta;
  const int sh = blockIdx.x / blocks_per, rb = blockIdx.x % blocks_per;
  const int s = sh / H, h = sh % H;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* p = smem_p + (size_t)warp * Tk;
  const act_t* kb = k + (size_t)s * Tk * k_ld + h * hd;
  const act_t* vb = v + (size_t)s * Tk * v_ld + h * hd;
  for (int i = rb * kRowsPerCta + warp; i < Tq && i < (rb + 1) * kRowsPerCta; i += kAttnWarps) {
    const act_t* qi = q + ((size_t)s * Tq + i) * q_ld + h * hd;
    float mx = -INFINITY;
    for (int j = lane; j < Tk; j += 32) {
      const float sc = dot_row16(qi, kb + (size_t)j * k_ld, hd) * scale;
      p[j] = sc;
      mx = fmaxf(mx, sc);
    }
    mx = warp_max(mx);
    float sum = 0.f;
    for (int j = lane; j < Tk; j += 32) { const float e = expf(p[j] - mx); p[j] = e; sum += e; }
    sum = warp_sum(sum);
    const float inv = 1.f / sum;
    __syncwarp();
    for (int d = lane; d < hd; d += 32) {
      float acc = 0.f;
      for (int j = 0; j < Tk; ++j) acc += p[j] * act2f(vb[(size_t)j * v_ld + d]);
      o[((size_t)s * Tq + i) * o_ld + h * hd + d] = f2act(acc * inv);
    }
    if (lane == 0) lse[((size_t)s * H + h) * Tq + i] = mx + logf(sum);
    __syncwarp();
  }
}

__global__ void __launch_bounds__(32 * kAttnWarps)
attn_bwd_dq_kernel(const act_t* __restrict__ q, int q_ld, const act_t* __restrict__ k, int k_ld, const act_t* __restrict__ v,
                   int v_ld, const float* __restrict__ d_o, int do_ld, const float* __restrict__ lse,
                   float* __restrict__ dsum, float* __restrict__ dq, int dq_ld, int H, int hd, int Tq, int Tk, float scale) {
  extern __shared__ float smem_p[];            // [kAttnWarps][2][Tk]: p_j, then p_j dP_j -> dS_j
  const int blocks_per = (Tq + kRowsPerCta - 1) / kRowsPerCta;
  const int sh = blockIdx.x / blocks_per, rb = blockIdx.x % blocks_per;
  const int s = sh / H, h = sh % H;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* pp = smem_p + (size_t)warp * 2 * Tk;
  float* ds = pp + Tk;
  const act_t* kb = k + (size_t)s * Tk * k_ld + h * hd;
  const act_t* vb = v + (size_t)s * Tk * v_ld + h * hd;
  for (int i = rb * kRowsPerCta + warp; i < Tq && i < (rb + 1) * kRowsPerCta; i += kAttnWarps) {
    const act_t* qi = q + ((size_t)s * Tq + i) * q_ld + h * hd;
    const float* doi = d_o + ((size_t)s * Tq + i) * do_ld + h * hd;
    const float l = lse[((size_t)s * H + h) * Tq + i];
    float dacc = 0.f;
    for (int j = lane; j < Tk; j += 32) {
      const float pj = expf(dot_row16(qi, kb + (size_t)j * k_ld, hd) * scale - l);
      const float dp = dot_row_f32_16(doi, vb + (size_t)j * v_ld, hd);
      pp[j] = pj;
      ds[j] = pj * dp;
      dacc += pj * dp;
    }
    const float D = warp_sum(dacc);
    if (lane == 0) dsum[((size_t)s * H + h) * Tq + i] = D;
    for (int j = lane; j < Tk; j += 32) ds[j] = (ds[j] - pp[j] * D) * scale;     // dS_j = p_j (dP_j - D_i) * scale
    __syncwarp();
    for (int d = lane; d < hd; d += 32) {
      float acc = 0.f;
      for (int j = 0; j < Tk; ++j) acc += ds[j] * act2f(kb[(size_t)j * k_ld + d]);
      dq[((size_t)s * Tq + i) * dq_ld + h * hd + d] += acc;
    }
    __syncwarp();
  }
}

__global__ void __launch_bounds__(32 * kAttnWarps)
attn_bwd_dkv_kernel(const act_t* __restrict__ q, int q_ld, const act_t* __restrict__ k, int k_ld, const act_t* __restrict__ v,
                    int v_ld, const float* __restrict__ d_o, int do_ld, const float* __restrict__ lse,
                    const float* __restrict__ dsum, float* __restrict__ dk, int dk_ld, float* __restrict__ dv, int dv_ld,
                    int H, int hd, int Tq, int Tk, float scale) {
  extern __shared__ float smem_p[];            // [kAttnWarps][2][Tq]: p_ij and dS_ij of the warp's key row
  const int blocks_per = (Tk + kRowsPerCta - 1) / kRowsPerCta;
  const int sh = blockIdx.x / blocks_per, rb = blockIdx.x % blocks_per;
  const int s = sh / H, h = sh % H;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* pp = smem_p + (size_t)warp * 2 * Tq;
  float* ds = pp + Tq;
  const act_t* qb = q + (size_t)s * Tq * q_ld + h * hd;
  const float* dob = d_o + (size_t)s * Tq * do_ld + h * hd;
  const float* lb = lse + ((size_t)s * H + h) * Tq;
  const float* Db = dsum + ((size_t)s * H + h) * Tq;
  for (int j = rb * kRowsPerCta + warp; j < Tk && j < (rb + 1) * kRowsPerCta; j += kAttnWarps) {
    const act_t* kj = k + ((size_t)s * Tk + j) * k_ld + h * hd;
    const act_t* vj = v + ((size_t)s * Tk + j) * v_ld + h * hd;
    for (int i = lane; i < Tq; i += 32) {
      const float pij = expf(dot_row16(qb + (size_t)i * q_ld, kj, hd) * scale - lb[i]);
      const float dp = dot_row_f32_16(dob + (size_t)i * do_ld, vj, hd);
      pp[i] = pij;
      ds[i] = pij * (dp - Db[i]) * scale;
    }
    __syncwarp();
    for (int d = lane; d < hd; d += 32) {
      float ak = 0.f, av = 0.f;
      for (int i = 0; i < Tq; ++i) {
        ak += ds[i] * act2f(qb[(size_t)i * q_ld + d]);
        av += pp[i] * dob[(size_t)i * do_ld + d];
      }
      dk[((size_t)s * Tk + j) * dk_ld + h * hd + d] += ak;
      dv[((size_t)s * Tk + j) * dv_ld + h * hd + d] += av;
    }
    __syncwarp();
  }
}

// ---------------------------------------------------------------------------------------------------------------
// BCE-with-logits (mean over all elements, nn.BCEWithLogitsLoss default): loss and scaled d loss / d logit
// ---------------------------------------------------------------------------------------------------------------
__global__ void bce_logits_kernel(const float* __restrict__ logits, const float* __restrict__ labels, int n,
                                  float* __restrict__ loss, float* __restrict__ dlogits, float grad_scale) {
  __shared__ float part[32];
  float acc = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const float x = logits[i], y = labels[i];
    acc += fmaxf(x, 0.f) - x * y + log1pf(expf(-fabsf(x)));
    dlogits[i] = (1.f / (1.f + expf(-x)) - y) * grad_scale / n;
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int w = 0; w < (blockDim.x >> 5); ++w) t += part[w];
    *loss = t / n;
  }
}

}  // namespace

// ---------------------------------------------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------------------------------------------
int train_cast_scale(const float* in, act_t* out, size_t n, float scale, cudaStream_t s) {
  if (n == 0) return 0;
  cast_scale_kernel<<<blocks_for(n), kThreads, 0, s>>>(in, out, n, scale);
  VITED_CUDA_OK(cudaGetLastError());
  return 0;
}
int train_act_axpby(const act_t* x, float* y, size_t n, float alpha, float beta, cudaStream_t s) {
  if (n == 0) return 0;
  act_axpby_kernel<<<blocks_for(n), kThreads, 0, s>>>(x, y, n, alpha, beta);
  VITED_CUDA_OK(cudaGetLastError());
  return 0;
}
int train_f32_axpy(const float* x, float* y, size_t n, float alpha, cudaStream_t s) {
  if (n == 0) return 0;
  f32_axpy_kernel<<<blocks_for(n), kThreads, 0, s>>>(x, y, n, alpha);
  VITED_CUDA_OK(cudaGetLastError());
  return 0;
}
int train_transpose(const void* in, int in_is_f32, int ld_in, act_t* out, int ld_out, int R, int C, float scale,
                    cudaStream_t s) {
  VITED_CHECK(ld_out >= R && ld_in >= C, "transpose: bad leading dimensions");
  if (R == 0 || C == 0) return 0;
  dim3 grid((C + 31) / 32, (ld_out + 31) / 32), block(32, 8);
  if (in_is_f32) transpose_kernel<float><<<grid, block, 0, s>>>((const float*)in, ld_in, out, ld_out, R, C, scale);
  else transpose_kernel<act_t><<<grid, block, 0, s>>>((const act_t*)in, ld_in, out, ld_out, R, C, scale);
  VITED_CUDA_OK(cudaGetLastError());
  return 0;
}
int train_ln_forward(const float* x, const float* w, const float* b, act_t* h, float* stats, int R, int D, float eps,
                     cudaStream_t s) {
  if (R == 0) return 0;
  ln_fwd_kernel<<<blocks_for((size_t)R * 32), kThreads, 0, s>>>(x, w, b, h, stats, R, D, eps);
  VITED_CUDA_OK(cudaGetLastError());
  return 0;
}
int train_ln_backward(const float* dh, const float* x, const float* stats, const float* w, float* dx, float* dw, float* db,
                      int R, int D, float alpha, cudaStream_t s) {
  if (R == 0) return 0;
  VITED_CHECK((size_t)2 * D * 4 <= 48 * 1024, "ln_backward: D=%d too large", D);
  ln_bwd_kernel<<<blocks_for((size_t)R * 32, kThreads, 148 * 2), kThreads, 2 * D * sizeof(float), s>>>(dh, x, stats, w, dx, dw,
                                                                                                     db, R, D, alpha);
  VITED_CUDA_OK(cudaGetLastError());
  return 0;
}
int train_gelu_forward(const act_t* z, act_t* a, size_t n, cudaStream_t s) {
  if (n == 0) return 0;
  gelu_fwd_kernel<<<blocks_for(n), kThreads, 0, s>>>(z, a, n);
  VITED_CUDA_OK(cudaGetLastError());
  return 0;
}
int train_gelu_backward(const float* da, const act_t* z, float* dz, size_t n, cudaStream_t s) {
  if (n == 0) return 0;
  gelu_bwd_kernel<<<blocks_for(n), kThreads, 0, s>>>(da, z, dz, n);
  VITED_CUDA_OK(cudaGetLastError());
  return 0;
}
int train_colsum(const float* dy, float* db, int R, int N, float alpha, cudaStream_t s) {
  if (R == 0 || N == 0) return 0;
  VITED_CHECK(N % 4 == 0 && (reinterpret_cast<uintptr_t>(dy) & 15) == 0, "colsum: N=%d must be a multiple of 4, dy 16-byte aligned", N);
  int gy = (R + 127) / 128;                    // ~16 rows per thread
  if (gy > 148 * 4) gy = 148 * 4;
  dim3 grid((N + 127) / 128, gy), block(32, 8);
  colsum_kernel<<<grid, block, 0, s>>>(dy, db, R, N, alpha);
  VITED_CUDA_OK(cudaGetLastError());
  return 0;
}
int train_gather_rows(const float* in, const int* idx, float* out, int n_blocks, int rows_per, int in_block_stride,
                      int in_row_off, int out_block_stride, int out_row_off, int D, int accumulate, cudaStream_t s) {
  const size_t total = (size_t)n_blocks * rows_per * D;
  if (total == 0) return 0;
  gather_rows_kernel<<<blocks_for(total), kThreads, 0, s>>>(in, idx, out, n_blocks, rows_per, in_block_stride, in_row_off,
                                                           out_block_stride, out_row_off, D, accumulate);
  VITED_CUDA_OK(cudaGetLastError());
  return 0;
}
int train_scatter_add_rows(const float* src, const int* idx, float* dst, int n_blocks, int rows_per, int src_block_stride,
                           int src_row_off, int dst_block_stride, int dst_row_off, int D, float alpha, cudaStream_t s) {
  const size_t total = (size_t)n_blocks * rows_per * D;
  if (total == 0) return 0;
  scatter_add_rows_kernel<<<blocks_for(total), kThreads, 0, s>>>(src, idx, dst, n_blocks, rows_per, src_block_stride,
                                                                src_row_off, dst_block_stride, dst_row_off, D, alpha);
  VITED_CUDA_OK(cudaGetLastError());
  return 0;
}
int train_col2im(const float* dcol, float* dimages, int B, int C, int S, int p, cudaStream_t s) {
  VITED_CHECK(B >= 0 && C > 0 && p > 0 && p % 4 == 0 && S % p == 0,
              "train col2im: patch size %d must be a multiple of 4 and divide img size %d (B %d, C %d)", p, S, B, C);
  VITED_CHECK((reinterpret_cast<uintptr_t>(dcol) | reinterpret_cast<uintptr_t>(dimages)) % 16 == 0,
              "train col2im: dcol and dimages must be 16-byte aligned");
  const size_t total = (size_t)B * (S / p) * (S / p) * (C * p * p / 4);
  if (total == 0) return 0;
  col2im_kernel<<<blocks_for(total), kThreads, 0, s>>>(dcol, dimages, B, C, S, p);
  VITED_CUDA_OK(cudaGetLastError());
  return 0;
}
int train_attention(int backward, const act_t* q, int q_ld, const act_t* k, int k_ld, const act_t* v, int v_ld, act_t* o,
                    int o_ld, float* lse, const float* d_o, int do_ld, float* dsum, float* dq, int dq_ld, float* dk, int dk_ld,
                    float* dv, int dv_ld, int n_seq, int H, int hd, int Tq, int Tk, float scale, cudaStream_t s, int* flag) {
  if (n_seq == 0) return 0;
  static const int simt = [] { const char* e = getenv("VITED_TRAIN_ATTN_SIMT"); return e ? atoi(e) : 0; }();
  VITED_CHECK(hd % 8 == 0 && q_ld % 8 == 0 && k_ld % 8 == 0 && v_ld % 8 == 0, "train attention: head_dim / strides must be multiples of 8");
  VITED_CHECK(((reinterpret_cast<uintptr_t>(q) | reinterpret_cast<uintptr_t>(k) | reinterpret_cast<uintptr_t>(v)) & 15) == 0,
              "train attention: q / k / v must be 16-byte aligned");
  if (!simt && train_attention_wmma_supported(hd)) {
    VITED_CHECK(o && lse && o_ld % 8 == 0, "train attention: the tensor-core path needs o (also in the backward pass) and lse");
    if (backward)
      VITED_CHECK(d_o && dsum && dq && dk && dv && do_ld % 4 == 0 && (reinterpret_cast<uintptr_t>(d_o) & 15) == 0,
                  "train attention backward: bad arguments");
    return train_attention_wmma(backward, q, q_ld, k, k_ld, v, v_ld, o, o_ld, lse, d_o, do_ld, dsum, dq, dq_ld, dk, dk_ld, dv,
                                dv_ld, n_seq, H, hd, Tq, Tk, scale, s, flag);
  }
  const int tmax = Tq > Tk ? Tq : Tk;
  const size_t smem = (size_t)kAttnWarps * 2 * tmax * sizeof(float);
  VITED_CHECK(smem <= 200 * 1024, "train attention: %d tokens need %zu bytes of shared memory", tmax, smem);
  static PerDeviceOnce once;
  if (once.first()) {
    VITED_CUDA_OK(cudaFuncSetAttribute(attn_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    VITED_CUDA_OK(cudaFuncSetAttribute(attn_bwd_dq_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    VITED_CUDA_OK(cudaFuncSetAttribute(attn_bwd_dkv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  }
  const int qblocks = n_seq * H * ((Tq + kRowsPerCta - 1) / kRowsPerCta);
  const int kblocks = n_seq * H * ((Tk + kRowsPerCta - 1) / kRowsPerCta);
  if (!backward) {
    VITED_CHECK(o && lse, "train attention forward: null output");
    attn_fwd_kernel<<<qblocks, 32 * kAttnWarps, (size_t)kAttnWarps * Tk * sizeof(float), s>>>(q, q_ld, k, k_ld, v, v_ld, o, o_ld,
                                                                                              lse, H, hd, Tq, Tk, scale);
  } else {
    VITED_CHECK(d_o && lse && dsum && dq && dk && dv && do_ld % 4 == 0 && (reinterpret_cast<uintptr_t>(d_o) & 15) == 0,
                "train attention backward: bad arguments");
    attn_bwd_dq_kernel<<<qblocks, 32 * kAttnWarps, (size_t)kAttnWarps * 2 * Tk * sizeof(float), s>>>(
        q, q_ld, k, k_ld, v, v_ld, d_o, do_ld, lse, dsum, dq, dq_ld, H, hd, Tq, Tk, scale);
    VITED_CUDA_OK(cudaGetLastError());
    attn_bwd_dkv_kernel<<<kblocks, 32 * kAttnWarps, (size_t)kAttnWarps * 2 * Tq * sizeof(float), s>>>(
        q, q_ld, k, k_ld, v, v_ld, d_o, do_ld, lse, dsum, dk, dk_ld, dv, dv_ld, H, hd, Tq, Tk, scale);
  }
  VITED_CUDA_OK(cudaGetLastError());
  return 0;
}
int train_bce_logits(const float* logits, const float* labels, int n, float* loss, float* dlogits, float grad_scale,
                     cudaStream_t s) {
  VITED_CHECK(n >= 1, "bce: empty batch");
  bce_logits_kernel<<<1, 256, 0, s>>>(logits, labels, n, loss, dlogits, grad_scale);
  VITED_CUDA_OK(cudaGetLastError());
  return 0;
}

}  // namespace vited
