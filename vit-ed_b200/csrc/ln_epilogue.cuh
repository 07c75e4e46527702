// LayerNorm arithmetic of the full-row epilogues in gemm_ln.cu and mlp_ln.cu (and of mlp_ln.cu's cross-projection
// prologue). Two threads own one row: each holds one NW-column half in registers / TMEM. Each half gets shifted one-pass
// statistics (pivot c0 = the half's first element); Chan's formula combines the two halves; then the row is normalised
// 8 columns at a time into packed 16-bit values. All arithmetic is in packed fp32 pairs (FADD2 / FFMA2): the epilogue
// passes are issue bound, and the pairs halve their arithmetic instructions.
#pragma once
#include "common.cuh"

namespace vited {

// v = acc + (b + x) for 4 columns: the residual add of a GEMM accumulator, its bias and the residual stream
__device__ __forceinline__ float4 ln_resid4(const uint32_t* acc, float4 b, float4 x) {
  float4 v;
  f2_unpack(f2_add(f2_from_bits(acc[0], acc[1]), f2_add(f2_pack(b.x, b.y), f2_pack(x.x, x.y))), v.x, v.y);
  f2_unpack(f2_add(f2_from_bits(acc[2], acc[3]), f2_add(f2_pack(b.z, b.w), f2_pack(x.z, x.w))), v.z, v.w);
  return v;
}

// shifted one-pass statistics of N columns of a row half: s += sum(v - c0), ss += sum((v - c0)^2)
template <int N>
__device__ __forceinline__ void ln_accum_stats(const uint32_t (&v)[N], float c0, float& s, float& ss) {
  uint64_t s2[2] = {0ull, 0ull}, q2[2] = {0ull, 0ull};                 // four independent chains each
  const uint64_t nc0 = f2_dup(-c0);
#pragma unroll
  for (int i = 0; i < N / 2; ++i) {
    const uint64_t d = f2_add(f2_from_bits(v[2 * i], v[2 * i + 1]), nc0);
    s2[i & 1] = f2_add(s2[i & 1], d);
    q2[i & 1] = f2_fma(d, d, q2[i & 1]);
  }
  float s4[4], q4[4];
  f2_unpack(s2[0], s4[0], s4[1]); f2_unpack(s2[1], s4[2], s4[3]);
  f2_unpack(q2[0], q4[0], q4[1]); f2_unpack(q2[1], q4[2], q4[3]);
  s += (s4[0] + s4[1]) + (s4[2] + s4[3]);
  ss += (q4[0] + q4[1]) + (q4[2] + q4[3]);
}

// Mean and 1 / sqrt(var + eps) of a 2 * NW-column row from the statistics (s, ss, c0) of this thread's half (Chan's
// combination). The halves meet through shared memory: this thread writes (mean, M2) of its half to `mine` and reads the
// partner's from `other` after named barrier `bar`, which kBarThreads threads (both threads of the row among them) reach.
template <int NW, int kBarThreads>
__device__ __forceinline__ void ln_row_stats(float2* mine, const float2* other, int bar, float s, float ss, float c0,
                                             float eps, uint64_t& nmean2, uint64_t& rstd2) {
  const float inv_n = 1.f / NW;
  const float mean_a = c0 + s * inv_n, m2_a = ss - s * s * inv_n;
  *mine = make_float2(mean_a, m2_a);
  asm volatile("bar.sync %0, %1;" ::"r"(bar), "n"(kBarThreads) : "memory");
  const float2 o = *other;
  const float dm = o.x - mean_a;
  const float mean = 0.5f * (mean_a + o.x);
  const float var = (m2_a + o.y + dm * dm * (0.5f * NW)) * (1.f / (2 * NW));
  const float rstd = rsqrtf(fmaxf(var, 0.f) + eps);
  nmean2 = f2_dup(-mean);
  rstd2 = f2_dup(rstd);
}

// (v - mean) * rstd * g + b of 8 columns as packed 16-bit values; g_a / bt_a: shared-window addresses of the first
// column's LayerNorm weight and bias
__device__ __forceinline__ uint4 ln_normalise8(const uint32_t* v, uint32_t g_a, uint32_t bt_a, uint64_t nmean2,
                                               uint64_t rstd2) {
  const float4 g0 = lds_f4(g_a);
  const float4 g1 = lds_f4(g_a + 16);
  const float4 t0 = lds_f4(bt_a);
  const float4 t1 = lds_f4(bt_a + 16);
  float y[8];
  f2_unpack(f2_fma(f2_mul(f2_add(f2_from_bits(v[0], v[1]), nmean2), rstd2), f2_pack(g0.x, g0.y), f2_pack(t0.x, t0.y)), y[0], y[1]);
  f2_unpack(f2_fma(f2_mul(f2_add(f2_from_bits(v[2], v[3]), nmean2), rstd2), f2_pack(g0.z, g0.w), f2_pack(t0.z, t0.w)), y[2], y[3]);
  f2_unpack(f2_fma(f2_mul(f2_add(f2_from_bits(v[4], v[5]), nmean2), rstd2), f2_pack(g1.x, g1.y), f2_pack(t1.x, t1.y)), y[4], y[5]);
  f2_unpack(f2_fma(f2_mul(f2_add(f2_from_bits(v[6], v[7]), nmean2), rstd2), f2_pack(g1.z, g1.w), f2_pack(t1.z, t1.w)), y[6], y[7]);
  uint4 pk;
  pk.x = pack_act(y[0], y[1]);
  pk.y = pack_act(y[2], y[3]);
  pk.z = pack_act(y[4], y[5]);
  pk.w = pack_act(y[6], y[7]);
  return pk;
}

}  // namespace vited
