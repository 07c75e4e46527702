// HBM-bound row kernels of the ViT-ED scoring path: patch im2col, token assembly (pos-embed / cls), fused
// residual-add + LayerNorm, final norm + head, plus a plain SIMT GEMM kept as an on-device debugging reference.
// One warp owns one token row (D = 384 -> three float4 per lane), loads are 16-byte and fully coalesced.
#include "kernels.h"

namespace vited {

// ------------------------------------------------------------------------------------------------------------
// im2col for Conv2d(kernel = stride = p)  (timm PatchEmbed; called from models/vision_transformer.py:383,391)
// token t = gy*G + gx covers pixels [gy*p:(gy+1)*p, gx*p:(gx+1)*p]; column = c*p*p + py*p + px.
// ------------------------------------------------------------------------------------------------------------
__global__ void im2col_kernel(const float* __restrict__ img, act_t* __restrict__ out, int B, int C, int S, int p,
                              const int* __restrict__ items) {
  const int G = S / p;
  const int K = C * p * p;
  const int segs_per_row = K / 4;  // 4 consecutive px per thread (p % 4 == 0)
  const size_t total = (size_t)B * G * G * segs_per_row;
  for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const int seg = (int)(idx % segs_per_row);
    const size_t row = idx / segs_per_row;
    const int col = seg * 4;
    const int c = col / (p * p);
    const int py = (col / p) % p;
    const int px = col % p;
    const int t = (int)(row % (G * G));
    const int b = (int)(row / (G * G));
    const size_t sb = items != nullptr ? (size_t)items[b] : (size_t)b;   // source image
    const int gy = t / G, gx = t % G;
    const float4 v = *reinterpret_cast<const float4*>(img + ((sb * C + c) * S + (gy * p + py)) * S + gx * p + px);
    uint2 pk;
    pk.x = pack_act(v.x, v.y);
    pk.y = pack_act(v.z, v.w);
    *reinterpret_cast<uint2*>(out + row * K + col) = pk;
  }
}

int im2col_patches(const float* images, act_t* out, int B, int C, int S, int p, cudaStream_t stream, const int* items) {
  VITED_CHECK(p % 4 == 0 && S % p == 0, "im2col: patch size %d must be a multiple of 4 and divide img size %d", p, S);
  const size_t total = (size_t)B * (S / p) * (S / p) * (C * p * p / 4);
  int blocks = (int)((total + 255) / 256);
  if (blocks > 148 * 16) blocks = 148 * 16;
  if (blocks < 1) blocks = 1;
  im2col_kernel<<<blocks, 256, 0, stream>>>(images, out, B, C, S, p, items);
  VITED_CUDA_OK(cudaGetLastError());
  return 0;
}

// The same patch matrix straight from the decoded bytes [B, S, S, C] (HWC uint8), with the normalisation of
// normalize_u8_kernel (ToTensor + Normalize(.5, .5), hisfrag.py:89-93) folded in. A byte has 256 values, so every
// block first evaluates that arithmetic once per value into a shared table of 16-bit results (rounded by pack_act,
// as im2col_kernel rounds): the output is bit-identical to normalize_u8 followed by im2col_patches.
// `items` non-null: output image b is read from image items[b] (the engine's gathered batches).
// One thread = one pixel row of one patch: P*C contiguous bytes (48 at P = 16), loaded as VB-byte vectors and
// de-interleaved in registers, then P 16-bit values per channel stored contiguously. gx runs fastest across a warp,
// so a warp reads whole pixel rows and every thread writes whole 32-byte sectors.
template <int P, int C, int VB>
__global__ void __launch_bounds__(256) im2col_u8_kernel(const uint8_t* __restrict__ img, act_t* __restrict__ out,
                                                        int B, int S, const int* __restrict__ items) {
  __shared__ uint16_t lut[256];
  for (int v = threadIdx.x; v < 256; v += blockDim.x) {
    const float f = __fdiv_rn(__fsub_rn(__fdiv_rn((float)v, 255.0f), 0.5f), 0.5f);
    lut[v] = (uint16_t)(pack_act(f, f) & 0xffffu);
  }
  __syncthreads();
  constexpr int NB = P * C;             // bytes of one patch pixel row
  constexpr int K = C * P * P;
  static_assert(NB % VB == 0 && NB % 4 == 0 && P % 4 == 0, "patch row must split into whole vectors");
  const int G = S / P;
  const size_t total = (size_t)B * S * G;   // (b, gy, py, gx), gx fastest
  for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const int gx = (int)(idx % G);
    const size_t by = idx / G;              // b * S + gy * P + py: the pixel row
    const int y = (int)(by % S);
    const size_t b = by / S;
    const int gy = y / P, py = y % P;
    uint32_t w[NB / 4];
    const size_t sb = items != nullptr ? (size_t)items[b] : b;   // source image
    const uint8_t* src = img + ((sb * S + y) * S + (size_t)gx * P) * C;
#pragma unroll
    for (int k = 0; k < NB / VB; ++k) {
      if constexpr (VB == 16) {
        const uint4 v = *reinterpret_cast<const uint4*>(src + k * 16);
        w[4 * k] = v.x; w[4 * k + 1] = v.y; w[4 * k + 2] = v.z; w[4 * k + 3] = v.w;
      } else if constexpr (VB == 8) {
        const uint2 v = *reinterpret_cast<const uint2*>(src + k * 8);
        w[2 * k] = v.x; w[2 * k + 1] = v.y;
      } else {
        w[k] = *reinterpret_cast<const uint32_t*>(src + k * 4);
      }
    }
    const size_t row = (b * G + gy) * G + gx;
    act_t* dst = out + row * K + py * P;
#pragma unroll
    for (int c = 0; c < C; ++c) {
      uint32_t o[P / 2];
#pragma unroll
      for (int px = 0; px < P; px += 2) {
        const int i0 = px * C + c, i1 = (px + 1) * C + c;     // byte of (px, c) inside the loaded row
        const uint32_t lo = lut[(w[i0 >> 2] >> (8 * (i0 & 3))) & 0xffu];
        const uint32_t hi = lut[(w[i1 >> 2] >> (8 * (i1 & 3))) & 0xffu];
        o[px / 2] = lo | (hi << 16);
      }
      act_t* d = dst + c * P * P;
#pragma unroll
      for (int k = 0; k < P / 8; ++k)
        *reinterpret_cast<uint4*>(d + 8 * k) = make_uint4(o[4 * k], o[4 * k + 1], o[4 * k + 2], o[4 * k + 3]);
      if constexpr (P % 8 != 0) *reinterpret_cast<uint2*>(d + P - 4) = make_uint2(o[P / 2 - 2], o[P / 2 - 1]);
    }
  }
}

int im2col_u8_patches(const uint8_t* images, act_t* out, int B, int C, int S, int p, cudaStream_t stream,
                      const int* items) {
  VITED_CHECK(B >= 0 && p > 0 && S % p == 0, "im2col_u8: patch size %d must divide img size %d", p, S);
  const size_t total = (size_t)B * S * (S / p);
  if (total == 0) return 0;
  int blocks = (int)((total + 255) / 256);
  if (blocks > 148 * 16) blocks = 148 * 16;
  // a pixel row of one patch starts at a multiple of p*C bytes; the vector width must divide that and the pointer
  const uintptr_t a = (uintptr_t)images;
#define VITED_IM2COL_U8(P_, C_, VB_)                                                                    \
  if (p == P_ && C == C_) {                                                                             \
    VITED_CHECK(a % VB_ == 0, "im2col_u8: images must be %d-byte aligned for patch %d", VB_, P_);       \
    im2col_u8_kernel<P_, C_, VB_><<<blocks, 256, 0, stream>>>(images, out, B, S, items);                \
    VITED_CUDA_OK(cudaGetLastError());                                                                  \
    return 0;                                                                                           \
  }
  VITED_IM2COL_U8(16, 3, 16)
  VITED_IM2COL_U8(8, 3, 8)
  VITED_IM2COL_U8(32, 3, 16)
  VITED_IM2COL_U8(4, 3, 4)
#undef VITED_IM2COL_U8
  set_error("im2col_u8: no kernel for patch size %d with %d channels (built for 4, 8, 16, 32 with 3)", p, C);
  return 1;
}

// ------------------------------------------------------------------------------------------------------------
// x0 = patch tokens + pos_embed[:, 1:]  (vision_transformer.py:378-380);  cls row = cls_token + pos_embed[:, 0]
// (timm _pos_embed, called at :392).  Split layout: B*Np patch rows, then B cls rows.
// ------------------------------------------------------------------------------------------------------------
__global__ void assemble_kernel(const act_t* __restrict__ tok, const float* __restrict__ pos,
                                const float* __restrict__ cls, float* __restrict__ x, int B, int Np, int D,
                                int with_cls) {
  const int D4 = D / 4;
  const size_t n_patch_rows = (size_t)B * Np;
  const size_t rows = n_patch_rows + (with_cls ? B : 0);
  const size_t total = rows * D4;
  for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const int d = (int)(idx % D4) * 4;
    const size_t row = idx / D4;
    float4 o;
    if (row < n_patch_rows) {
      const int t = (int)(row % Np);
      const uint2 tk = *reinterpret_cast<const uint2*>(tok + row * D + d);
      const float2 a = unpack_act(tk.x), b = unpack_act(tk.y);
      const float4 pe = *reinterpret_cast<const float4*>(pos + (size_t)(1 + t) * D + d);
      o = make_float4(a.x + pe.x, a.y + pe.y, b.x + pe.z, b.y + pe.w);
    } else {
      const float4 c4 = *reinterpret_cast<const float4*>(cls + d);
      const float4 pe = *reinterpret_cast<const float4*>(pos + d);
      o = make_float4(c4.x + pe.x, c4.y + pe.y, c4.z + pe.z, c4.w + pe.w);
    }
    *reinterpret_cast<float4*>(x + row * D + d) = o;
  }
}

int assemble_tokens(const act_t* tok, const float* pos_embed, const float* cls_token, float* x, int B, int n_patch,
                    int D, int with_cls, cudaStream_t stream) {
  VITED_CHECK(D % 4 == 0, "assemble: D=%d must be a multiple of 4", D);
  const size_t total = ((size_t)B * n_patch + (with_cls ? B : 0)) * (D / 4);
  int blocks = (int)((total + 255) / 256);
  if (blocks > 148 * 16) blocks = 148 * 16;
  if (blocks < 1) blocks = 1;
  assemble_kernel<<<blocks, 256, 0, stream>>>(tok, pos_embed, cls_token, x, B, n_patch, D, with_cls);
  VITED_CUDA_OK(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------------------------------------------------
// fused residual add (+ gather from the per-item cache) + LayerNorm(eps 1e-6) -> fp16 GEMM operand.
// Mirrors `x = x + sub_block(...)` followed by the next block's `normX(x)` (vision_transformer.py:124-127, 268-272).
// One warp per row; NV = D / 128 float4 per lane.
// ------------------------------------------------------------------------------------------------------------
template <int NV>
__global__ void __launch_bounds__(256) resid_ln_kernel(ResidLnArgs a) {
  const int lane = threadIdx.x & 31;
  const int D = a.D;
  const size_t n_patch_rows = (size_t)a.n_seq * a.n_patch;
  const size_t rows = n_patch_rows + (a.has_cls ? a.n_seq : 0);
  const size_t warps_total = ((size_t)gridDim.x * blockDim.x) >> 5;
  for (size_t row = (((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5); row < rows; row += warps_total) {
    const float* src = a.x + row * D;
    if (a.gather_src != nullptr) {
      size_t srow;
      if (row < n_patch_rows) {
        const int s = (int)(row / a.n_patch);
        const int t = (int)(row % a.n_patch);
        srow = (size_t)(a.gather_idx[s] - a.gather_off) * a.n_patch + t;
      } else {
        srow = (size_t)a.n_src_seq * a.n_patch + (a.gather_idx[row - n_patch_rows] - a.gather_off);
      }
      src = a.gather_src + srow * D;
    }
    float4 v[NV];
#pragma unroll
    for (int i = 0; i < NV; ++i) v[i] = *reinterpret_cast<const float4*>(src + i * 128 + lane * 4);
    if (a.delta != nullptr) {
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        const uint2 dl = *reinterpret_cast<const uint2*>(a.delta + row * D + i * 128 + lane * 4);
        const float2 d0 = unpack_act(dl.x), d1 = unpack_act(dl.y);
        v[i].x += d0.x; v[i].y += d0.y; v[i].z += d1.x; v[i].w += d1.y;
      }
    }
    if (a.write_x) {
#pragma unroll
      for (int i = 0; i < NV; ++i) *reinterpret_cast<float4*>(a.x + row * D + i * 128 + lane * 4) = v[i];
    }
    if (a.ln_w != nullptr) {
      float s = 0.f;
#pragma unroll
      for (int i = 0; i < NV; ++i) s += v[i].x + v[i].y + v[i].z + v[i].w;
      const float mean = warp_sum(s) / (float)D;
      float ss = 0.f;
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        const float dx = v[i].x - mean, dy = v[i].y - mean, dz = v[i].z - mean, dw = v[i].w - mean;
        ss += dx * dx + dy * dy + dz * dz + dw * dw;
      }
      const float rstd = rsqrtf(warp_sum(ss) / (float)D + a.eps);
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        const float4 w4 = __ldg(reinterpret_cast<const float4*>(a.ln_w + i * 128 + lane * 4));
        const float4 b4 = __ldg(reinterpret_cast<const float4*>(a.ln_b + i * 128 + lane * 4));
        uint2 pk;
        pk.x = pack_act((v[i].x - mean) * rstd * w4.x + b4.x, (v[i].y - mean) * rstd * w4.y + b4.y);
        pk.y = pack_act((v[i].z - mean) * rstd * w4.z + b4.z, (v[i].w - mean) * rstd * w4.w + b4.w);
        *reinterpret_cast<uint2*>(a.h + row * D + i * 128 + lane * 4) = pk;
      }
    }
  }
}

// generic-D variant (any D % 4 == 0, e.g. the reference's tiny test config EMBED_DIM 32): lane-strided float4.
__global__ void __launch_bounds__(256) resid_ln_generic_kernel(ResidLnArgs a) {
  const int lane = threadIdx.x & 31;
  const int D = a.D;
  const int D4 = D / 4;
  const size_t n_patch_rows = (size_t)a.n_seq * a.n_patch;
  const size_t rows = n_patch_rows + (a.has_cls ? a.n_seq : 0);
  const size_t warps_total = ((size_t)gridDim.x * blockDim.x) >> 5;
  for (size_t row = (((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5); row < rows; row += warps_total) {
    const float* src = a.x + row * D;
    if (a.gather_src != nullptr) {
      size_t srow;
      if (row < n_patch_rows) {
        srow = (size_t)(a.gather_idx[row / a.n_patch] - a.gather_off) * a.n_patch + (row % a.n_patch);
      } else {
        srow = (size_t)a.n_src_seq * a.n_patch + (a.gather_idx[row - n_patch_rows] - a.gather_off);
      }
      src = a.gather_src + srow * D;
    }
    float s = 0.f;
    for (int i = lane; i < D4; i += 32) {
      float4 v = *reinterpret_cast<const float4*>(src + i * 4);
      if (a.delta != nullptr) {
        const uint2 dl = *reinterpret_cast<const uint2*>(a.delta + row * D + i * 4);
        const float2 d0 = unpack_act(dl.x), d1 = unpack_act(dl.y);
        v.x += d0.x; v.y += d0.y; v.z += d1.x; v.w += d1.y;
      }
      // keep the updated row in x (also used as scratch for the second pass when !write_x is never requested
      // together with gather/delta by the engine)
      if (a.write_x) *reinterpret_cast<float4*>(a.x + row * D + i * 4) = v;
      s += v.x + v.y + v.z + v.w;
    }
    if (a.ln_w == nullptr) continue;
    __syncwarp();
    const float* xr = a.write_x ? (a.x + row * D) : src;
    const float mean = warp_sum(s) / (float)D;
    float ss = 0.f;
    for (int i = lane; i < D4; i += 32) {
      const float4 v = *reinterpret_cast<const float4*>(xr + i * 4);
      const float dx = v.x - mean, dy = v.y - mean, dz = v.z - mean, dw = v.w - mean;
      ss += dx * dx + dy * dy + dz * dz + dw * dw;
    }
    const float rstd = rsqrtf(warp_sum(ss) / (float)D + a.eps);
    for (int i = lane; i < D4; i += 32) {
      const float4 v = *reinterpret_cast<const float4*>(xr + i * 4);
      const float4 w4 = __ldg(reinterpret_cast<const float4*>(a.ln_w + i * 4));
      const float4 b4 = __ldg(reinterpret_cast<const float4*>(a.ln_b + i * 4));
      uint2 pk;
      pk.x = pack_act((v.x - mean) * rstd * w4.x + b4.x, (v.y - mean) * rstd * w4.y + b4.y);
      pk.y = pack_act((v.z - mean) * rstd * w4.z + b4.z, (v.w - mean) * rstd * w4.w + b4.w);
      *reinterpret_cast<uint2*>(a.h + row * D + i * 4) = pk;
    }
  }
}

int resid_ln(const ResidLnArgs& a, cudaStream_t stream) {
  VITED_CHECK(a.D % 4 == 0, "resid_ln: D=%d must be a multiple of 4", a.D);
  const size_t rows = (size_t)a.n_seq * a.n_patch + (a.has_cls ? a.n_seq : 0);
  if (rows == 0) return 0;
  size_t blocks = (rows + 7) / 8;
  if (blocks > 148 * 32) blocks = 148 * 32;
  if (a.D == 384) {
    resid_ln_kernel<3><<<(int)blocks, 256, 0, stream>>>(a);
  } else if (a.D == 768) {
    resid_ln_kernel<6><<<(int)blocks, 256, 0, stream>>>(a);
  } else {
    // the generic kernel re-reads the row from x; it needs write_x whenever the row is modified
    VITED_CHECK(a.write_x || (a.delta == nullptr), "resid_ln(generic D=%d): delta requires write_x", a.D);
    resid_ln_generic_kernel<<<(int)blocks, 256, 0, stream>>>(a);
  }
  VITED_CUDA_OK(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------------------------------------------------
// final LayerNorm on the cls row + Linear(D, C) head (vision_transformer.py:400, :417 -> timm forward_head).
// Only row 0 of every sequence feeds the head, so the norm is applied to the cls rows alone. One warp per pair.
// ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) head_kernel(HeadArgs a) {
  const int lane = threadIdx.x & 31;
  const int D = a.D;
  const size_t warps_total = ((size_t)gridDim.x * blockDim.x) >> 5;
  for (size_t p = (((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5); p < (size_t)a.P; p += warps_total) {
    const float* xr = a.x + p * D;
    float s = 0.f;
    for (int d = lane; d < D; d += 32) {
      float v = xr[d];
      if (a.delta != nullptr) v += act2f(a.delta[p * D + d]);
      s += v;
    }
    const float mean = warp_sum(s) / (float)D;
    float ss = 0.f;
    for (int d = lane; d < D; d += 32) {
      float v = xr[d];
      if (a.delta != nullptr) v += act2f(a.delta[p * D + d]);
      ss += (v - mean) * (v - mean);
    }
    const float rstd = rsqrtf(warp_sum(ss) / (float)D + a.eps);
    size_t obase;
    if (a.out_pos != nullptr) {
      obase = (size_t)a.out_pos[p] * a.C;
    } else if (a.ci != nullptr) {
      obase = ((size_t)(a.ci[p] - a.row_begin) * a.n_items + a.xj[p]) * a.C;
    } else {
      obase = p * a.C;
    }
    for (int c = 0; c < a.C; ++c) {
      float acc = 0.f;
      for (int d = lane; d < D; d += 32) {
        float v = xr[d];
        if (a.delta != nullptr) v += act2f(a.delta[p * D + d]);
        const float y = (v - mean) * rstd * __ldg(a.ln_w + d) + __ldg(a.ln_b + d);
        acc += y * __ldg(a.head_w + (size_t)c * D + d);
      }
      acc = warp_sum(acc);
      if (lane == 0) a.out[obase + c] = acc + __ldg(a.head_b + c);
    }
  }
}

int head_logits(const HeadArgs& a, cudaStream_t stream) {
  if (a.P == 0) return 0;
  size_t blocks = ((size_t)a.P + 7) / 8;
  if (blocks > 148 * 32) blocks = 148 * 32;
  head_kernel<<<(int)blocks, 256, 0, stream>>>(a);
  VITED_CUDA_OK(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------------------------------------------------
// pair lists of a block of grid rows, generated where they are consumed (no host vectors, no upload, no sync)
// ------------------------------------------------------------------------------------------------------------
__host__ __device__ size_t pair_list_count(int mode, int r0, int r1, int ca, int cb) {
  const size_t nr = (size_t)(r1 - r0);
  if (mode == 0) {     // nr * (cb - ca) minus the diagonal entries inside the window
    const int lo = r0 > ca ? r0 : ca, hi = r1 < cb ? r1 : cb;
    return nr * (size_t)(cb - ca) - (size_t)(hi > lo ? hi - lo : 0);
  }
  if (mode == 1) {     // rows i < ca see the whole window, rows i in [ca, cb) see [i, cb)
    const int below = (r1 < ca ? r1 : ca) - r0;
    const int lo = r0 > ca ? r0 : ca, hi = r1 < cb ? r1 : cb;
    size_t n = below > 0 ? (size_t)below * (size_t)(cb - ca) : 0;
    if (hi > lo) n += (size_t)(hi - lo) * (size_t)cb - ((size_t)lo + hi - 1) * (size_t)(hi - lo) / 2;
    return n;
  }
  return nr;
}

__global__ void __launch_bounds__(256) pair_list_kernel(int mode, int r0, int r1, int ca, int cb, int* __restrict__ ci,
                                                        int* __restrict__ xj) {
  for (int i = r0 + (int)blockIdx.x; i < r1; i += (int)gridDim.x) {
    if (mode == 2) {
      if (threadIdx.x == 0) { ci[i - r0] = i - r0; xj[i - r0] = i - r0; }
      continue;
    }
    const size_t off = pair_list_count(mode, r0, i, ca, cb);
    const int len = (int)pair_list_count(mode, i, i + 1, ca, cb);
    const int j0 = (mode == 0 || i < ca) ? ca : i;
    const bool skip_diag = (mode == 0) && i >= ca;
    for (int t = threadIdx.x; t < len; t += blockDim.x) {
      const int j = j0 + t + ((skip_diag && j0 + t >= i) ? 1 : 0);
      ci[off + t] = i - r0;
      xj[off + t] = j;
    }
  }
}

int pair_list(int mode, int r0, int r1, int ca, int cb, int* ci, int* xj, cudaStream_t stream) {
  VITED_CHECK(mode >= 0 && mode <= 2 && r0 >= 0 && r0 <= r1 && ca >= 0 && ca <= cb, "pair_list: bad arguments");
  if (r1 == r0) return 0;
  int blocks = r1 - r0;
  if (blocks > 148 * 8) blocks = 148 * 8;
  pair_list_kernel<<<blocks, 256, 0, stream>>>(mode, r0, r1, ca, cb, ci, xj);
  VITED_CUDA_OK(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------------------------------------------------
// small converters
// ------------------------------------------------------------------------------------------------------------
__global__ void f32_to_act_kernel(const float* __restrict__ in, act_t* __restrict__ out, size_t n) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    out[i] = f2act(in[i]);
}
int f32_to_act(const float* in, act_t* out, size_t n, cudaStream_t stream) {
  if (n == 0) return 0;
  size_t blocks = (n + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  f32_to_act_kernel<<<(int)blocks, 256, 0, stream>>>(in, out, n);
  VITED_CUDA_OK(cudaGetLastError());
  return 0;
}

__global__ void add_delta_out_kernel(const float* __restrict__ x, const act_t* __restrict__ delta,
                                     float* __restrict__ out, size_t n) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    out[i] = x[i] + act2f(delta[i]);
}
int add_delta_out(const float* x, const act_t* delta, float* out, size_t rows, int D, cudaStream_t stream) {
  const size_t n = rows * D;
  if (n == 0) return 0;
  size_t blocks = (n + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  add_delta_out_kernel<<<(int)blocks, 256, 0, stream>>>(x, delta, out, n);
  VITED_CUDA_OK(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------------------------------------------------
// debugging reference GEMM (SIMT, fp32 accumulate). Same contract as the tcgen05 kernel; never used by default.
// ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) gemm_simt_kernel(const act_t* __restrict__ A, const act_t* __restrict__ W,
                                                        const float* __restrict__ bias, act_t* __restrict__ C, int M,
                                                        int N, int K, int act) {
  __shared__ float sA[16][64 + 1];
  __shared__ float sW[16][64 + 1];
  const int tx = threadIdx.x % 16, ty = threadIdx.x / 16;
  const int m0 = blockIdx.y * 64, n0 = blockIdx.x * 64;
  float acc[4][4] = {};
  for (int k0 = 0; k0 < K; k0 += 16) {
    for (int i = threadIdx.x; i < 64 * 16; i += 256) {
      const int r = i / 16, kk = i % 16;
      sA[kk][r] = (m0 + r < M && k0 + kk < K) ? act2f(A[(size_t)(m0 + r) * K + k0 + kk]) : 0.f;
      sW[kk][r] = (n0 + r < N && k0 + kk < K) ? act2f(W[(size_t)(n0 + r) * K + k0 + kk]) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < 16; ++kk) {
      float a[4], w[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { a[i] = sA[kk][ty * 4 + i]; w[i] = sW[kk][tx * 4 + i]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] += a[i] * w[j];
    }
    __syncthreads();
  }
  for (int i = 0; i < 4; ++i)
    for (int j = 0; j < 4; ++j) {
      const int m = m0 + ty * 4 + i, n = n0 + tx * 4 + j;
      if (m < M && n < N) {
        float v = acc[i][j] + (bias ? bias[n] : 0.f);
        if (act == ACT_GELU) v = gelu_erf(v);
        C[(size_t)m * N + n] = f2act(v);
      }
    }
}

int gemm_simt(const act_t* A, const act_t* W, const float* bias, act_t* C, int M, int N, int K, int act,
              cudaStream_t stream) {
  dim3 grid((N + 63) / 64, (M + 63) / 64);
  gemm_simt_kernel<<<grid, 256, 0, stream>>>(A, W, bias, C, M, N, K, act);
  VITED_CUDA_OK(cudaGetLastError());
  return 0;
}

}  // namespace vited
