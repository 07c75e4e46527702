// Softmax attention of the training step on the warp-level tensor cores (wmma m16n16k16, fp32 accumulation): flash-style
// forward and backward, nothing quadratic stored, no atomics. Plain token layout (see train_ops.cu).
//   forward  : per (sequence, head, 64 query rows): S = Q K^T per 64-key block, online softmax, O = P V, lse per row
//   D        : D_i = do_i . o_i  (= sum_j p_ij dP_ij), one warp per (row, head)
//   backward : dK, dV per (sequence, head, 64 key rows): S^T = K Q^T, dP^T = V dO^T per 64-query block,
//              P^T = exp(S^T * scale - lse), dS^T = P^T (dP^T - D) * scale, dV += P^T dO, dK += dS^T Q;
//              dQ per (sequence, head, 64 query rows): the same quantities untransposed, dQ += dS K.
// Every operand of an MMA is a 16-bit tile in shared memory, every elementwise step (softmax, dS) reads the fp32
// accumulator tile back from shared memory: simple and robust rather than fast -- this is the training side (SURVEY 8f
// row 1), not the scoring hot path, whose attention runs on tcgen05 (attention_tc.cu). It replaces the one-warp-per-row
// fp32 kernels of train_ops.cu (kept as the reference implementation, VITED_TRAIN_ATTN_SIMT=1): 4.0 s -> see
// profiles/README.md per Hisfrag20 step.
#include "kernels.h"
#include <mma.h>

namespace vited {

namespace {

using namespace nvcuda;

constexpr int BR = 64;           // rows of the block a CTA owns (16 per warp)
constexpr int BC = 64;           // rows of the streamed block
constexpr int LDS_F = BC + 4;    // leading dimension of fp32 [16 x 64] tiles (floats)
constexpr int LDS_H = BC + 8;    // leading dimension of 16-bit [16 x 64] tiles
constexpr int kWarps = 4;

template <int HD> struct Ld { static constexpr int H = HD + 8; static constexpr int F = HD + 4; };

// [rows x HD] 16-bit tile from a strided global matrix (zero beyond n_valid rows)
template <int HD>
__device__ __forceinline__ void load_tile16(act_t* dst, const act_t* src, int ld, int n_valid, int tid, int nthreads) {
  constexpr int CH = HD / 8;     // 16-byte chunks per row
  for (int i = tid; i < BR * CH; i += nthreads) {
    const int r = i / CH, c = i % CH;
    uint4 v = make_uint4(0, 0, 0, 0);
    if (r < n_valid) v = *reinterpret_cast<const uint4*>(src + (size_t)r * ld + c * 8);
    *reinterpret_cast<uint4*>(dst + r * Ld<HD>::H + c * 8) = v;
  }
}
// same from an fp32 matrix (converted to 16 bits)
template <int HD>
__device__ __forceinline__ void load_tile32(act_t* dst, const float* src, int ld, int n_valid, int tid, int nthreads) {
  constexpr int CH = HD / 4;
  for (int i = tid; i < BR * CH; i += nthreads) {
    const int r = i / CH, c = i % CH;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (r < n_valid) v = *reinterpret_cast<const float4*>(src + (size_t)r * ld + c * 4);
    act_t* d = dst + r * Ld<HD>::H + c * 4;
    d[0] = f2act(v.x); d[1] = f2act(v.y); d[2] = f2act(v.z); d[3] = f2act(v.w);
  }
}

typedef wmma::fragment<wmma::matrix_a, 16, 16, 16, act_t, wmma::row_major> FragA;
typedef wmma::fragment<wmma::matrix_b, 16, 16, 16, act_t, wmma::col_major> FragBc;   // B(k, n) = M[n][k]: "times M^T"
typedef wmma::fragment<wmma::matrix_b, 16, 16, 16, act_t, wmma::row_major> FragBr;   // B(k, n) = M[k][n]: "times M"
typedef wmma::fragment<wmma::accumulator, 16, 16, 16, float> FragC;

// out[16 x 64] (fp32, shared) = A[16 x HD] * M[64 x HD]^T
template <int HD>
__device__ __forceinline__ void mm_abt(float* out, const act_t* a, const act_t* m) {
#pragma unroll
  for (int n = 0; n < BC / 16; ++n) {
    FragC c;
    wmma::fill_fragment(c, 0.f);
#pragma unroll
    for (int k = 0; k < HD / 16; ++k) {
      FragA fa;
      FragBc fb;
      wmma::load_matrix_sync(fa, a + k * 16, Ld<HD>::H);
      wmma::load_matrix_sync(fb, m + n * 16 * Ld<HD>::H + k * 16, Ld<HD>::H);
      wmma::mma_sync(c, fa, fb, c);
    }
    wmma::store_matrix_sync(out + n * 16, c, LDS_F, wmma::mem_row_major);
  }
}

// acc[HD / 16] (+)= P[16 x 64] (16-bit, shared) * M[64 x HD]
template <int HD>
__device__ __forceinline__ void mm_pm(FragC (&acc)[HD / 16], const act_t* p, const act_t* m) {
#pragma unroll
  for (int k = 0; k < BC / 16; ++k) {
    FragA fa;
    wmma::load_matrix_sync(fa, p + k * 16, LDS_H);
#pragma unroll
    for (int n = 0; n < HD / 16; ++n) {
      FragBr fb;
      wmma::load_matrix_sync(fb, m + k * 16 * Ld<HD>::H + n * 16, Ld<HD>::H);
      wmma::mma_sync(acc[n], fa, fb, acc[n]);
    }
  }
}

template <int HD>
struct FwdSmem {
  static constexpr size_t kWarpBytes = 16 * LDS_F * 4 + 16 * LDS_H * 2 + 2 * 16 * Ld<HD>::F * 4;   // S, P, O, PV
  static constexpr size_t BYTES = 3 * BR * Ld<HD>::H * 2 + kWarps * kWarpBytes + 128;
};

template <int HD>
__global__ void __launch_bounds__(32 * kWarps)
attn_wmma_fwd_kernel(const act_t* __restrict__ q, int q_ld, const act_t* __restrict__ k, int k_ld, const act_t* __restrict__ v,
                     int v_ld, act_t* __restrict__ o, int o_ld, float* __restrict__ lse, int H, int Tq, int Tk, float scale) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  act_t* sQ = reinterpret_cast<act_t*>(smem_raw);
  act_t* sK = sQ + BR * Ld<HD>::H;
  act_t* sV = sK + BC * Ld<HD>::H;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint8_t* wbase = reinterpret_cast<uint8_t*>(sV + BC * Ld<HD>::H) + warp * FwdSmem<HD>::kWarpBytes;
  float* sS = reinterpret_cast<float*>(wbase);
  act_t* sP = reinterpret_cast<act_t*>(sS + 16 * LDS_F);
  float* sO = reinterpret_cast<float*>(sP + 16 * LDS_H);
  float* sT = sO + 16 * Ld<HD>::F;
  const int qblocks = (Tq + BR - 1) / BR;
  const int sh = blockIdx.x / qblocks, qb = blockIdx.x % qblocks;
  const int s = sh / H, h = sh % H;
  const int q0 = qb * BR;
  load_tile16<HD>(sQ, q + ((size_t)s * Tq + q0) * q_ld + h * HD, q_ld, Tq - q0, threadIdx.x, 32 * kWarps);
  for (int i = lane; i < 16 * Ld<HD>::F; i += 32) sO[i] = 0.f;
  // lane -> (row of the warp's 16, half of the 64 columns): two lanes share a row
  const int r = lane >> 1, half = lane & 1;
  float m_run = -INFINITY, l_run = 0.f;
  for (int k0 = 0; k0 < Tk; k0 += BC) {
    __syncthreads();                                        // the previous block's K / V tiles are no longer read
    load_tile16<HD>(sK, k + ((size_t)s * Tk + k0) * k_ld + h * HD, k_ld, Tk - k0, threadIdx.x, 32 * kWarps);
    load_tile16<HD>(sV, v + ((size_t)s * Tk + k0) * v_ld + h * HD, v_ld, Tk - k0, threadIdx.x, 32 * kWarps);
    __syncthreads();
    mm_abt<HD>(sS, sQ + warp * 16 * Ld<HD>::H, sK);
    __syncwarp();
    // online softmax of this lane's half row
    float mx = -INFINITY;
    const float* srow = sS + r * LDS_F + half * 32;
#pragma unroll 8
    for (int j = 0; j < 32; ++j)
      if (k0 + half * 32 + j < Tk) mx = fmaxf(mx, srow[j] * scale);
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
    const float m_new = fmaxf(m_run, mx);
    const float alpha = (m_run == -INFINITY) ? 0.f : expf(m_run - m_new);
    float sum = 0.f;
    act_t* prow = sP + r * LDS_H + half * 32;
#pragma unroll 8
    for (int j = 0; j < 32; ++j) {
      float pj = 0.f;
      if (k0 + half * 32 + j < Tk) pj = expf(srow[j] * scale - m_new);
      const act_t ph = f2act(pj);
      prow[j] = ph;
      sum += act2f(ph);                                     // the row sum of what the MMA will actually multiply
    }
    sum += __shfl_xor_sync(0xffffffffu, sum, 1);
    l_run = l_run * alpha + sum;
    m_run = m_new;
    __syncwarp();
    FragC acc[HD / 16];
#pragma unroll
    for (int n = 0; n < HD / 16; ++n) wmma::fill_fragment(acc[n], 0.f);
    mm_pm<HD>(acc, sP, sV);
#pragma unroll
    for (int n = 0; n < HD / 16; ++n) wmma::store_matrix_sync(sT + n * 16, acc[n], Ld<HD>::F, wmma::mem_row_major);
    __syncwarp();
    for (int d = half * (HD / 2); d < (half + 1) * (HD / 2); ++d)
      sO[r * Ld<HD>::F + d] = sO[r * Ld<HD>::F + d] * alpha + sT[r * Ld<HD>::F + d];
    __syncwarp();
  }
  const int qi = q0 + warp * 16 + r;
  if (qi < Tq) {
    const float inv = 1.f / l_run;
    act_t* orow = o + ((size_t)s * Tq + qi) * o_ld + h * HD;
    for (int d = half * (HD / 2); d < (half + 1) * (HD / 2); ++d) orow[d] = f2act(sO[r * Ld<HD>::F + d] * inv);
    if (half == 0) lse[((size_t)s * H + h) * Tq + qi] = m_run + logf(l_run);
  }
}

// D[s, h, i] = sum_d do[s, i, h, d] * o[s, i, h, d]
__global__ void attn_dsum_kernel(const float* __restrict__ d_o, int do_ld, const act_t* __restrict__ o, int o_ld,
                                 float* __restrict__ dsum, int n_seq, int H, int hd, int Tq) {
  const int lane = threadIdx.x & 31;
  const size_t total = (size_t)n_seq * H * Tq;
  const size_t warps = ((size_t)gridDim.x * blockDim.x) >> 5;
  for (size_t w = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < total; w += warps) {
    const int i = (int)(w % Tq);
    const int h = (int)((w / Tq) % H);
    const int s = (int)(w / ((size_t)Tq * H));
    float acc = 0.f;
    for (int d = lane; d < hd; d += 32)
      acc += d_o[((size_t)s * Tq + i) * do_ld + h * hd + d] * act2f(o[((size_t)s * Tq + i) * o_ld + h * hd + d]);
    acc = warp_sum(acc);
    if (lane == 0) dsum[w] = acc;
  }
}

template <int HD>
struct BwdSmem {
  // own block + streamed block: two [64 x HD] 16-bit tiles each; per warp: two fp32 [16 x 64] tiles, two 16-bit ones,
  // and an fp32 [16 x HD] staging tile for the results; lse / D of the 64 streamed (or own) query rows
  static constexpr size_t kWarpBytes = 2 * 16 * LDS_F * 4 + 2 * 16 * LDS_H * 2 + 16 * Ld<HD>::F * 4;
  static constexpr size_t BYTES = 4 * BR * Ld<HD>::H * 2 + kWarps * kWarpBytes + 2 * BR * 4 + 128;
};

// CHK: *flag = 1 when a dS value is out of the 16-bit range (|dS| can reach about 2 |dO_i| max_j |V_j| scale even
// when dO is in range); the flag is the last parameter so that the unchecked form keeps its parameter layout
template <bool CHK>
__device__ __forceinline__ void report_out_of_range(bool bad, int* flag) {
  if constexpr (CHK) {
    if (__any_sync(0xffffffffu, bad) && (threadIdx.x & 31) == 0) *flag = 1;
  }
}

// dK, dV of 64 key rows (16 per warp); streams the query blocks
template <int HD, bool CHK>
__global__ void __launch_bounds__(32 * kWarps)
attn_wmma_bwd_dkv_kernel(const act_t* __restrict__ q, int q_ld, const act_t* __restrict__ k, int k_ld,
                         const act_t* __restrict__ v, int v_ld, const float* __restrict__ d_o, int do_ld,
                         const float* __restrict__ lse, const float* __restrict__ dsum, float* __restrict__ dk, int dk_ld,
                         float* __restrict__ dv, int dv_ld, int H, int Tq, int Tk, float scale, int* __restrict__ flag) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  act_t* sK = reinterpret_cast<act_t*>(smem_raw);
  act_t* sV = sK + BR * Ld<HD>::H;
  act_t* sQ = sV + BR * Ld<HD>::H;
  act_t* sDO = sQ + BC * Ld<HD>::H;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint8_t* wbase = reinterpret_cast<uint8_t*>(sDO + BC * Ld<HD>::H) + warp * BwdSmem<HD>::kWarpBytes;
  float* sS = reinterpret_cast<float*>(wbase);
  float* sDP = sS + 16 * LDS_F;
  act_t* sP = reinterpret_cast<act_t*>(sDP + 16 * LDS_F);
  act_t* sDS = sP + 16 * LDS_H;
  float* sT = reinterpret_cast<float*>(sDS + 16 * LDS_H);
  float* sLse = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(sDO + BC * Ld<HD>::H) + kWarps * BwdSmem<HD>::kWarpBytes);
  float* sD = sLse + BC;
  const int kblocks = (Tk + BR - 1) / BR;
  const int sh = blockIdx.x / kblocks, kb = blockIdx.x % kblocks;
  const int s = sh / H, h = sh % H;
  const int k0 = kb * BR;
  load_tile16<HD>(sK, k + ((size_t)s * Tk + k0) * k_ld + h * HD, k_ld, Tk - k0, threadIdx.x, 32 * kWarps);
  load_tile16<HD>(sV, v + ((size_t)s * Tk + k0) * v_ld + h * HD, v_ld, Tk - k0, threadIdx.x, 32 * kWarps);
  FragC acc_dk[HD / 16], acc_dv[HD / 16];
#pragma unroll
  for (int n = 0; n < HD / 16; ++n) { wmma::fill_fragment(acc_dk[n], 0.f); wmma::fill_fragment(acc_dv[n], 0.f); }
  const int r = lane >> 1, half = lane & 1;
  const bool key_ok = k0 + warp * 16 + r < Tk;
  bool bad = false;
  for (int q0 = 0; q0 < Tq; q0 += BC) {
    __syncthreads();
    load_tile16<HD>(sQ, q + ((size_t)s * Tq + q0) * q_ld + h * HD, q_ld, Tq - q0, threadIdx.x, 32 * kWarps);
    load_tile32<HD>(sDO, d_o + ((size_t)s * Tq + q0) * do_ld + h * HD, do_ld, Tq - q0, threadIdx.x, 32 * kWarps);
    for (int i = threadIdx.x; i < BC; i += 32 * kWarps) {
      const bool ok = q0 + i < Tq;
      sLse[i] = ok ? lse[((size_t)s * H + h) * Tq + q0 + i] : 0.f;
      sD[i] = ok ? dsum[((size_t)s * H + h) * Tq + q0 + i] : 0.f;
    }
    __syncthreads();
    mm_abt<HD>(sS, sK + warp * 16 * Ld<HD>::H, sQ);        // S^T  [16 keys x 64 queries]
    mm_abt<HD>(sDP, sV + warp * 16 * Ld<HD>::H, sDO);      // dP^T
    __syncwarp();
#pragma unroll 8
    for (int j = 0; j < 32; ++j) {
      const int c = half * 32 + j;
      float p = 0.f, ds = 0.f;
      if (key_ok && q0 + c < Tq) {
        p = expf(sS[r * LDS_F + c] * scale - sLse[c]);
        ds = p * (sDP[r * LDS_F + c] - sD[c]) * scale;
        if constexpr (CHK) bad |= !(fabsf(ds) < kActRangeLimit);
      }
      sP[r * LDS_H + c] = f2act(p);
      sDS[r * LDS_H + c] = f2act(ds);
    }
    __syncwarp();
    mm_pm<HD>(acc_dv, sP, sDO);                             // dV += P^T dO
    mm_pm<HD>(acc_dk, sDS, sQ);                             // dK += dS^T Q
    __syncwarp();
  }
  const int kj = k0 + warp * 16 + r;
#pragma unroll
  for (int pass = 0; pass < 2; ++pass) {
#pragma unroll
    for (int n = 0; n < HD / 16; ++n)
      wmma::store_matrix_sync(sT + n * 16, pass == 0 ? acc_dk[n] : acc_dv[n], Ld<HD>::F, wmma::mem_row_major);
    __syncwarp();
    if (kj < Tk) {
      float* dst = (pass == 0 ? dk + ((size_t)s * Tk + kj) * dk_ld : dv + ((size_t)s * Tk + kj) * dv_ld) + h * HD;
      for (int d = half * (HD / 2); d < (half + 1) * (HD / 2); ++d) dst[d] += sT[r * Ld<HD>::F + d];
    }
    __syncwarp();
  }
  report_out_of_range<CHK>(bad, flag);
}

// dQ of 64 query rows (16 per warp); streams the key blocks
template <int HD, bool CHK>
__global__ void __launch_bounds__(32 * kWarps)
attn_wmma_bwd_dq_kernel(const act_t* __restrict__ q, int q_ld, const act_t* __restrict__ k, int k_ld,
                        const act_t* __restrict__ v, int v_ld, const float* __restrict__ d_o, int do_ld,
                        const float* __restrict__ lse, const float* __restrict__ dsum, float* __restrict__ dq, int dq_ld,
                        int H, int Tq, int Tk, float scale, int* __restrict__ flag) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  act_t* sQ = reinterpret_cast<act_t*>(smem_raw);
  act_t* sDO = sQ + BR * Ld<HD>::H;
  act_t* sK = sDO + BR * Ld<HD>::H;
  act_t* sV = sK + BC * Ld<HD>::H;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint8_t* wbase = reinterpret_cast<uint8_t*>(sV + BC * Ld<HD>::H) + warp * BwdSmem<HD>::kWarpBytes;
  float* sS = reinterpret_cast<float*>(wbase);
  float* sDP = sS + 16 * LDS_F;
  act_t* sDS = reinterpret_cast<act_t*>(sDP + 16 * LDS_F) + 16 * LDS_H;   // (the P tile of the layout is unused here)
  float* sT = reinterpret_cast<float*>(sDS + 16 * LDS_H);
  const int qblocks = (Tq + BR - 1) / BR;
  const int sh = blockIdx.x / qblocks, qb = blockIdx.x % qblocks;
  const int s = sh / H, h = sh % H;
  const int q0 = qb * BR;
  load_tile16<HD>(sQ, q + ((size_t)s * Tq + q0) * q_ld + h * HD, q_ld, Tq - q0, threadIdx.x, 32 * kWarps);
  load_tile32<HD>(sDO, d_o + ((size_t)s * Tq + q0) * do_ld + h * HD, do_ld, Tq - q0, threadIdx.x, 32 * kWarps);
  const int r = lane >> 1, half = lane & 1;
  const int qi = q0 + warp * 16 + r;
  const bool q_ok = qi < Tq;
  const float my_lse = q_ok ? lse[((size_t)s * H + h) * Tq + qi] : 0.f;
  const float my_d = q_ok ? dsum[((size_t)s * H + h) * Tq + qi] : 0.f;
  FragC acc[HD / 16];
#pragma unroll
  for (int n = 0; n < HD / 16; ++n) wmma::fill_fragment(acc[n], 0.f);
  bool bad = false;
  for (int k0 = 0; k0 < Tk; k0 += BC) {
    __syncthreads();
    load_tile16<HD>(sK, k + ((size_t)s * Tk + k0) * k_ld + h * HD, k_ld, Tk - k0, threadIdx.x, 32 * kWarps);
    load_tile16<HD>(sV, v + ((size_t)s * Tk + k0) * v_ld + h * HD, v_ld, Tk - k0, threadIdx.x, 32 * kWarps);
    __syncthreads();
    mm_abt<HD>(sS, sQ + warp * 16 * Ld<HD>::H, sK);        // S   [16 queries x 64 keys]
    mm_abt<HD>(sDP, sDO + warp * 16 * Ld<HD>::H, sV);      // dP
    __syncwarp();
#pragma unroll 8
    for (int j = 0; j < 32; ++j) {
      const int c = half * 32 + j;
      float ds = 0.f;
      if (q_ok && k0 + c < Tk) {
        const float p = expf(sS[r * LDS_F + c] * scale - my_lse);
        ds = p * (sDP[r * LDS_F + c] - my_d) * scale;
        if constexpr (CHK) bad |= !(fabsf(ds) < kActRangeLimit);
      }
      sDS[r * LDS_H + c] = f2act(ds);
    }
    __syncwarp();
    mm_pm<HD>(acc, sDS, sK);                                // dQ += dS K
    __syncwarp();
  }
#pragma unroll
  for (int n = 0; n < HD / 16; ++n) wmma::store_matrix_sync(sT + n * 16, acc[n], Ld<HD>::F, wmma::mem_row_major);
  __syncwarp();
  if (q_ok) {
    float* dst = dq + ((size_t)s * Tq + qi) * dq_ld + h * HD;
    for (int d = half * (HD / 2); d < (half + 1) * (HD / 2); ++d) dst[d] += sT[r * Ld<HD>::F + d];
  }
  report_out_of_range<CHK>(bad, flag);
}

template <int HD, bool CHK>
int launch_wmma(int backward, const act_t* q, int q_ld, const act_t* k, int k_ld, const act_t* v, int v_ld, act_t* o,
                int o_ld, float* lse, const float* d_o, int do_ld, float* dsum, float* dq, int dq_ld, float* dk, int dk_ld,
                float* dv, int dv_ld, int n_seq, int H, int Tq, int Tk, float scale, cudaStream_t s, int* flag) {
  static PerDeviceOnce once;
  if (once.first()) {
    VITED_CUDA_OK(cudaFuncSetAttribute(attn_wmma_fwd_kernel<HD>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FwdSmem<HD>::BYTES));
    VITED_CUDA_OK(cudaFuncSetAttribute(attn_wmma_bwd_dkv_kernel<HD, CHK>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)BwdSmem<HD>::BYTES));
    VITED_CUDA_OK(cudaFuncSetAttribute(attn_wmma_bwd_dq_kernel<HD, CHK>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)BwdSmem<HD>::BYTES));
  }
  const int qblocks = n_seq * H * ((Tq + BR - 1) / BR), kblocks = n_seq * H * ((Tk + BR - 1) / BR);
  if (!backward) {
    attn_wmma_fwd_kernel<HD><<<qblocks, 32 * kWarps, FwdSmem<HD>::BYTES, s>>>(q, q_ld, k, k_ld, v, v_ld, o, o_ld, lse, H, Tq, Tk, scale);
  } else {
    size_t rows = (size_t)n_seq * H * Tq;
    int blocks = (int)((rows + 7) / 8);
    if (blocks > 148 * 16) blocks = 148 * 16;
    attn_dsum_kernel<<<blocks, 256, 0, s>>>(d_o, do_ld, o, o_ld, dsum, n_seq, H, HD, Tq);
    VITED_CUDA_OK(cudaGetLastError());
    attn_wmma_bwd_dkv_kernel<HD, CHK><<<kblocks, 32 * kWarps, BwdSmem<HD>::BYTES, s>>>(q, q_ld, k, k_ld, v, v_ld, d_o, do_ld, lse, dsum,
                                                                                       dk, dk_ld, dv, dv_ld, H, Tq, Tk, scale, flag);
    VITED_CUDA_OK(cudaGetLastError());
    attn_wmma_bwd_dq_kernel<HD, CHK><<<qblocks, 32 * kWarps, BwdSmem<HD>::BYTES, s>>>(q, q_ld, k, k_ld, v, v_ld, d_o, do_ld, lse, dsum,
                                                                                      dq, dq_ld, H, Tq, Tk, scale, flag);
  }
  VITED_CUDA_OK(cudaGetLastError());
  return 0;
}

}  // namespace

bool train_attention_wmma_supported(int hd) { return hd == 32 || hd == 64; }

// o (16-bit, the forward output) is an INPUT of the backward pass here: D_i = do_i . o_i
int train_attention_wmma(int backward, const act_t* q, int q_ld, const act_t* k, int k_ld, const act_t* v, int v_ld, act_t* o,
                         int o_ld, float* lse, const float* d_o, int do_ld, float* dsum, float* dq, int dq_ld, float* dk,
                         int dk_ld, float* dv, int dv_ld, int n_seq, int H, int hd, int Tq, int Tk, float scale, cudaStream_t s,
                         int* flag) {
  auto* launch = hd == 32 ? (flag ? launch_wmma<32, true> : launch_wmma<32, false>)
                          : (flag ? launch_wmma<64, true> : launch_wmma<64, false>);
  return launch(backward, q, q_ld, k, k_ld, v, v_ld, o, o_ld, lse, d_o, do_ld, dsum, dq, dq_ld, dk, dk_ld, dv, dv_ld, n_seq, H,
                Tq, Tk, scale, s, flag);
}

}  // namespace vited
