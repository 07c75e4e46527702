// Shared device/host helpers for the ViT-ED all-pairs scoring kernels (sm_100a only).
// PTX wrappers: mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (alloc / mma / commit / ld), ldmatrix, mma.sync.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda.h>
#include <stdint.h>
#include <stdio.h>

namespace vited {

// The 16-bit type of every GEMM / attention operand and of every activation buffer. fp16 (11 significand bits) by
// default: it is the reference's own autocast dtype (config.py:216 AMP_ENABLE, fp16 GradScaler path) and gives ~6x
// smaller logit error against the fp32 reference than bf16 at the same speed and bytes (tests/analysis/
// sim_operand_dtype.py: max 1e-3 vs 6e-3..8e-3). Everything that can grow -- residual stream, LayerNorm statistics,
// softmax, accumulators -- stays fp32, and conversions saturate to +-65504 instead of producing inf.
// -DVITED_ACT_BF16=1 builds the bf16 variant (same kernels; used for the A/B error measurement).
#ifndef VITED_ACT_BF16
#define VITED_ACT_BF16 0
#endif
#if VITED_ACT_BF16
typedef __nv_bfloat16 act_t;
#else
typedef __half act_t;
#endif

// ---------------------------------------------------------------------------------------------
// host side error plumbing (no exceptions cross the C-ABI; see include/vited_b200.h)
// ---------------------------------------------------------------------------------------------
void set_error(const char* fmt, ...);
const char* get_error();

#define VITED_CUDA_OK(expr)                                                                     \
  do {                                                                                          \
    cudaError_t _e = (expr);                                                                    \
    if (_e != cudaSuccess) {                                                                    \
      vited::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e));   \
      return 1;                                                                                 \
    }                                                                                           \
  } while (0)

#define VITED_CHECK(cond, ...)                                                                  \
  do {                                                                                          \
    if (!(cond)) {                                                                              \
      vited::set_error(__VA_ARGS__);                                                            \
      return 1;                                                                                 \
    }                                                                                           \
  } while (0)

// One-time setup PER DEVICE: cudaFuncSetAttribute(MaxDynamicSharedMemorySize) and occupancy / SM-count queries apply to
// the current device only, and a process may hold engines on several GPUs (a handle is bound to one device). first()
// is true the first time it is called with a given device current. Callers serialise per the C-ABI contract.
struct PerDeviceOnce {
  unsigned long long done = 0;
  bool first() {
    int d = 0;
    cudaGetDevice(&d);
    const unsigned long long bit = 1ull << (d & 63);
    if (done & bit) return false;
    done |= bit;
    return true;
  }
};
int device_sm_count();   // SM count of the CURRENT device (cached per device); gemm_tc.cu

#ifdef __CUDACC__
// ---------------------------------------------------------------------------------------------
// small device helpers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// Explicit shared-memory accesses through 32-bit shared-window addresses. Pointers into the dynamic shared-memory
// carve-up lose their address space on the way through lambdas / arrays and compile to generic 64-bit LD.E / ST.E
// (address arithmetic in register pairs, slower path); the epilogue loops are latency / issue bound, so they use these.
__device__ __forceinline__ float4 lds_f4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ void sts_f4(uint32_t addr, float4 v) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void sts_u4(uint32_t addr, uint4 v) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

__device__ __forceinline__ uint32_t pack_act(float lo, float hi) {
#if VITED_ACT_BF16
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
#else
  uint32_t r;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
#endif
}

__device__ __forceinline__ float2 unpack_act(uint32_t u) {
#if VITED_ACT_BF16
  __nv_bfloat162 v = *reinterpret_cast<__nv_bfloat162*>(&u);
  return __bfloat1622float2(v);
#else
  __half2 v = *reinterpret_cast<__half2*>(&u);
  return __half22float2(v);
#endif
}

__device__ __forceinline__ float act2f(act_t v) {
#if VITED_ACT_BF16
  return __bfloat162float(v);
#else
  return __half2float(v);
#endif
}
__device__ __forceinline__ act_t f2act(float v) {
#if VITED_ACT_BF16
  return __float2bfloat16_rn(v);
#else
  return __float2half_rn(fminf(fmaxf(v, -65504.f), 65504.f));
#endif
}

// one lane of a converged warp (always the same one: lane 0 for a full mask). Issuing tcgen05.mma / commit under this
// predicate from WARP-UNIFORM code lets the compiler keep descriptors in uniform registers; issuing from a divergent
// `if (lane == 0)` block costs an ELECT / R2UR / BRA.U.ANY loop (~100 cycles) per MMA instruction.
__device__ __forceinline__ uint32_t elect_one_sync() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t"
      ".reg .b32 rx;\n\t"
      ".reg .pred px;\n\t"
      "elect.sync rx|px, %1;\n\t"
      "@px mov.s32 %0, 1;\n\t"
      "}\n"
      : "+r"(pred)
      : "r"(0xffffffffu));
  return pred;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// exact-erf GELU (timm Mlp default act_layer=nn.GELU, approximate='none')
__device__ __forceinline__ float gelu_erf(float x) {
  return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f));
}

// exact-erf GELU with ONE MUFU op: gelu(v) = max(v, 0) - 0.5*|v|*erfc(|v|/sqrt(2)), and erfc(a/sqrt(2)) = 2^(-Q(a)) with a
// cubic Q (all coefficients positive, so 2^(-Q) decays monotonically for any |v|) fitted minimax on the GELU value:
// |error| < 9e-5 everywhere, 1/50 of the fp16 rounding step of an O(1) activation (the result is stored as fp16).
// 6 FP32 ops + ex2.approx. The fc1 epilogue is instruction-issue bound (16 epilogue warps x 64 columns per tile), so
// every op counts: the degree-5 fit (6e-7) cost two more FMAs per element. (fit: tools/fit_gelu.py)
__device__ __forceinline__ float gelu_fast(float v) {
  const float a = fabsf(v);
  float q = fmaf(a, -0.0275597216f, -0.488495773f);
  q = fmaf(a, q, -1.140745f);
  q *= a;                                   // -Q(|v|)
  float e;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(q));
  return fmaf(-0.5f * a, e, fmaxf(v, 0.0f));
}

// ---------------------------------------------------------------------------------------------
// packed fp32 pairs (sm_100: FFMA2 / FADD2 process two fp32 values per issue slot) and the softmax exponentials
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t f2_pack(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void f2_unpack(uint64_t v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ uint64_t f2_fma(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ uint64_t f2_add(uint64_t a, uint64_t b) {
  uint64_t d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ uint64_t f2_mul(uint64_t a, uint64_t b) {
  uint64_t d;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ uint64_t f2_dup(float v) { return f2_pack(v, v); }
__device__ __forceinline__ uint64_t f2_from_bits(uint32_t lo, uint32_t hi) { return f2_pack(__uint_as_float(lo), __uint_as_float(hi)); }
__device__ __forceinline__ uint64_t f2_add_rm(uint64_t a, uint64_t b) {
  uint64_t d;
  asm("add.rm.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// 2^x of both halves for x <= 0 WITHOUT the MUFU pipe: floor(x) by the round-down magic add (the low mantissa bits of
// x + 1.5 * 2^23 are floor(x) in two's complement), a degree-3 minimax polynomial for 2^frac on [0, 1) (relative error
// 8.6e-5, a sixth of an fp16 rounding step; p(1) < 2, so the mantissa never carries) and the integer part added to the
// exponent field. 10 instructions per pair (2 FMNMX, 3 FADD2, 3 FFMA2, 2 LEA) against 2 MUFU.EX2 of 8 pipe cycles each.
__device__ __forceinline__ uint64_t ex2_poly2(uint64_t x2) {
  float x0, x1;
  f2_unpack(x2, x0, x1);
  x0 = fmaxf(x0, -126.f);
  x1 = fmaxf(x1, -126.f);
  const uint64_t x = f2_pack(x0, x1);
  const uint64_t xf = f2_add_rm(x, f2_pack(12582912.f, 12582912.f));
  const uint64_t fl = f2_add(xf, f2_pack(-12582912.f, -12582912.f));
  float f0, f1;
  f2_unpack(fl, f0, f1);
  const uint64_t fr = f2_add(x, f2_pack(-f0, -f1));
  uint64_t p = f2_fma(f2_pack(0.07706724107265472f, 0.07706724107265472f), fr, f2_pack(0.22764497995376587f, 0.22764497995376587f));
  p = f2_fma(p, fr, f2_pack(0.6951166391372681f, 0.6951166391372681f));
  p = f2_fma(p, fr, f2_pack(1.f, 1.f));
  float p0, p1, m0, m1;
  f2_unpack(p, p0, p1);
  f2_unpack(xf, m0, m1);
  return f2_pack(__uint_as_float(__float_as_uint(p0) + (__float_as_uint(m0) << 23)),
                 __uint_as_float(__float_as_uint(p1) + (__float_as_uint(m1) << 23)));
}
// TWICE the GELU of both halves (gelu_fast's approximation, same coefficients): 2 gelu(v) = v + |v| (1 - 2^(-Q(|v|))).
// |v| and -|v| are operand modifiers of FFMA2 / FMUL2, so a pair costs 2 FFMA2 + FMUL2 + 2 MUFU.EX2 + FFMA2 + FADD2 = 7
// issue slots against 14 for two gelu_fast calls. The factor 1/2 is left to the consumer: the fused MLP kernel
// multiplies the fc2 accumulator by 0.5 in the FMA that adds bias and residual (exact: a power of two).
__device__ __forceinline__ uint64_t gelu2x_fast2(uint64_t x2) {
  float x0, x1;
  f2_unpack(x2, x0, x1);
  const uint64_t a2 = f2_pack(fabsf(x0), fabsf(x1));
  uint64_t q = f2_fma(a2, f2_dup(-0.0275597216f), f2_dup(-0.488495773f));
  q = f2_fma(a2, q, f2_dup(-1.140745f));
  q = f2_mul(q, a2);                        // -Q(|v|)
  float q0, q1;
  f2_unpack(q, q0, q1);
  const uint64_t e2 = f2_pack(ex2_approx(q0), ex2_approx(q1));
  return f2_add(x2, f2_fma(f2_pack(-fabsf(x0), -fabsf(x1)), e2, a2));
}
// The exponentials of NP score pairs of one softmax row: pk[j] = fp16x2(2^(v[2j] sl2 + mneg), 2^(v[2j+1] sl2 + mneg)),
// probabilities accumulated into two packed sums (four chains). kExpPoly of every 8 pairs are computed with ex2_poly2
// on the FMA pipe, the rest with MUFU.EX2.
// Measured on B200 (profiles/r02b_softmax_variants.jsonl): long-sequence attention 0.742 ms scalar, 0.712 packed, 0.679 /
// 0.674 / 0.663 with 1 / 2 / 3 of 8; in the step 2 of 8 is best (power cap).
constexpr int kExpPoly = 2;
template <int NP>
__device__ __forceinline__ void softmax_exp_pairs(const uint32_t* v, float sl2, float mneg, uint32_t* pk, uint64_t (&sum2)[2]) {
  const uint64_t s2 = f2_pack(sl2, sl2), m2 = f2_pack(mneg, mneg);
#pragma unroll
  for (int j = 0; j < NP; ++j) {
    const uint64_t x = f2_fma(f2_pack(__uint_as_float(v[2 * j]), __uint_as_float(v[2 * j + 1])), s2, m2);
    uint64_t p;
    float p0, p1;
    if ((j & 7) < kExpPoly) {
      p = ex2_poly2(x);
      f2_unpack(p, p0, p1);
    } else {
      float x0, x1;
      f2_unpack(x, x0, x1);
      p0 = ex2_approx(x0);
      p1 = ex2_approx(x1);
      p = f2_pack(p0, p1);
    }
    sum2[j & 1] = f2_add(sum2[j & 1], p);
    pk[j] = pack_act(p0, p1);
  }
}

// ---------------------------------------------------------------------------------------------
// mbarrier
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// try_wait with a suspend-time hint: the waiting thread sleeps in hardware until the phase completes (or the hint, in
// ns, expires) instead of re-polling every ~80 cycles. Polling warps otherwise flood the MIO queue (ncu: MUFU / UTCMMA
// issue of the working warps stalls on `mio_throttle` behind tens of millions of SYNCS try-waits).
#ifndef VITED_MBAR_SUSPEND_NS
#define VITED_MBAR_SUSPEND_NS 20000
#endif
__device__ __forceinline__ uint32_t mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity), "r"((uint32_t)VITED_MBAR_SUSPEND_NS)
      : "memory");
  return ok;
}
// non-blocking probe (try_wait may suspend the thread for a system-dependent time; pollers of several barriers use this)
__device__ __forceinline__ uint32_t mbar_test_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok;
}
// Bounded wait: a protocol bug must trap (launch error on the host) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity, int tag) {
#ifdef VITED_JITTER
  // Timing fuzzer for the barrier protocols (-DVITED_JITTER): roughly one wait in four first sleeps 0..4 us, so
  // warps reach their waits in orders the production timing never produces. A protocol that relies on "the producer
  // cannot be that far ahead" shows up as a bounded-wait timeout or a wrong result in the kernel tests.
  {
    const uint32_t c = (uint32_t)clock64() * 2654435761u + (threadIdx.x >> 5) * 40503u + blockIdx.x * 9176u;
    if (((c >> 13) & 3u) == 0u) __nanosleep((c >> 17) & 4095u);
  }
#endif
  if (mbar_try_wait(bar, parity)) return;
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > 200000u) {  // each failed try sleeps up to 20 us: ~4 s
      printf("vited: mbarrier timeout tag=%d block=%d thread=%d parity=%u\n", tag, (int)blockIdx.x,
             (int)threadIdx.x, parity);
      __trap();
    }
  }
}

// ---------------------------------------------------------------------------------------------
// TMA
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* tm) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tm)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(const CUtensorMap* tm, uint64_t* bar, void* smem_dst, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tm)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
// L2 prefetch of one box (no shared-memory destination, no completion tracking): a later tma_load_2d of the same bytes
// then costs an L2 hit instead of an HBM round trip. Only worth it where L2 / HBM bandwidth is not the bound.
__device__ __forceinline__ void tma_prefetch_l2_2d(const CUtensorMap* tm, int c0, int c1) {
  asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global.tile [%0, {%1, %2}];" ::"l"(reinterpret_cast<uint64_t>(tm)),
               "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* tm, const void* smem_src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(tm)),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// ---------------------------------------------------------------------------------------------
// tcgen05 / TMEM
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_holder, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_holder)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem desc] * B[smem desc]; fp16 x fp16 -> fp32, issued by ONE thread.
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on an mbarrier once all previously issued tcgen05.mma of this thread have completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld_32x32b_x8(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
               : "memory");
}
// registers -> TMEM (each thread writes its own lane = tile row); used to hand softmax probabilities (packed fp16
// pairs, one 32-bit column = two consecutive K elements) to tcgen05.mma as the A operand
__device__ __forceinline__ void tmem_st_32x32b_x32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]),
      "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]),
      "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st_32x32b_x16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_32x32b_x8(uint32_t taddr, const uint32_t (&r)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(r[0]),
               "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld_32x32b_x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
// width-generic forms for the full-row epilogues, which exist with 32- and 16-column chunks (8 / 16 epilogue warps)
__device__ __forceinline__ void tmem_ld_cols(uint32_t taddr, uint32_t (&r)[32]) { tmem_ld_32x32b_x32(taddr, r); }
__device__ __forceinline__ void tmem_ld_cols(uint32_t taddr, uint32_t (&r)[16]) { tmem_ld_32x32b_x16(taddr, r); }
__device__ __forceinline__ void tmem_st_cols(uint32_t taddr, const uint32_t (&r)[32]) { tmem_st_32x32b_x32(taddr, r); }
__device__ __forceinline__ void tmem_st_cols(uint32_t taddr, const uint32_t (&r)[16]) { tmem_st_32x32b_x16(taddr, r); }
__device__ __forceinline__ void tmem_st_cols(uint32_t taddr, const uint32_t (&r)[8]) { tmem_st_32x32b_x8(taddr, r); }
// 16-byte chunk i of this lane's row inside a TMA box whose rows are ROWB bytes = the box's swizzle span
// (128B swizzle: chunk ^ (row & 7); 64B swizzle: chunk ^ ((row >> 1) & 3)); one lane = one row
template <int ROWB>
__device__ __forceinline__ uint32_t swz_chunk(int i, int lane) {
  static_assert(ROWB == 128 || ROWB == 64, "box rows of 128 or 64 bytes");
  return ROWB == 128 ? (uint32_t)(i ^ (lane & 7)) : (uint32_t)(i ^ ((lane >> 1) & 3));
}
// D[tmem] (+)= A[tmem, packed fp16 pairs] * B[smem desc]
__device__ __forceinline__ void umma_f16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}

// ---- CTA-pair (cta_group::2) variants: two SMs of one cluster share a 256-row tile --------------------------------
// In a cluster, a shared::cta address carries the CTA rank in bit 24; clearing it addresses the same offset in the
// leader CTA (rank 0) of the pair.
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_alloc_2cta(uint32_t* smem_holder, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_holder)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish_2cta() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_2cta(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// TMA load into THIS CTA's shared memory whose transaction bytes are counted on the LEADER CTA's mbarrier
__device__ __forceinline__ void tma_load_2d_2cta(const CUtensorMap* tm, uint64_t* bar, void* smem_dst, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tm)), "r"(smem_u32(bar) & kPeerBitMask), "r"(c0), "r"(c1)
      : "memory");
}
// D[tmem, both CTAs] (+)= A * B with M = 256 split over the pair; issued by ONE thread of the leader CTA
__device__ __forceinline__ void umma_f16_2cta(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// D[tmem, both CTAs] (+)= A[tmem, packed fp16 pairs, each CTA's own 128 rows] * B[smem desc, split over the pair]
__device__ __forceinline__ void umma_f16_ts_2cta(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc,
                                                  uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on the mbarrier at this shared-memory offset in BOTH CTAs once the issued cta_group::2 MMAs have completed
__device__ __forceinline__ void umma_commit_2cta(uint64_t* bar) {
  const uint16_t mask = 3;
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
          smem_u32(bar)),
      "h"(mask)
      : "memory");
}
// arrive on the LEADER CTA's copy of a barrier (from either CTA of the pair)
__device__ __forceinline__ void mbar_arrive_leader(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(smem_u32(bar) & kPeerBitMask) : "memory");
}

// K-major, 128-byte-swizzled shared-memory matrix descriptor (tile rows are 128 B = 64 fp16; 8-row groups are
// 1024 B apart). Field layout follows the PTX ISA "matrix descriptor" (start>>4 | LBO>>4 @16 | SBO>>4 @32 |
// version=1 @46 | swizzle mode @61, 2 = 128B).
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>(1) << 16;             // leading byte offset: unused for swizzled K-major
  d |= static_cast<uint64_t>(1024 >> 4) << 32;     // stride byte offset between 8-row core-matrix groups
  d |= static_cast<uint64_t>(1) << 46;             // descriptor version (Blackwell)
  d |= static_cast<uint64_t>(2) << 61;             // SWIZZLE_128B
  return d;
}
// The same descriptor split into its two 32-bit halves: the high word is a constant of the layout, the low word is
// (address >> 4) | LBO. An issuer loop keeps `lo` of stage 0 and adds stage * (stage bytes >> 4) and 2 * k per 16-wide
// k-step: one integer add per operand instead of rebuilding the 64-bit descriptor from the address every k-block (the
// issuer warp is a single dependent instruction stream; every instruction it does not execute is tensor-pipe time).
__device__ __forceinline__ uint32_t umma_desc_sw128_lo(uint32_t smem_addr) {
  return ((smem_addr & 0x3FFFFu) >> 4) | (1u << 16);
}
constexpr uint32_t kUmmaDescSw128Hi = (1024u >> 4) | (1u << 14) | (2u << 29);   // SBO 1024 B, version 1, SWIZZLE_128B
__device__ __forceinline__ uint64_t umma_desc_pack(uint32_t lo, uint32_t hi) {
  uint64_t d;
  asm("mov.b64 %0, {%1, %2};" : "=l"(d) : "r"(lo), "r"(hi));
  return d;
}
// General swizzled descriptor. swizzle_bytes 128 / 64: tile rows are that many bytes wide (what a TMA box with the same
// swizzle writes), 8-row groups are 8*swizzle_bytes apart (SBO). For a K-major operand the rows are M/N indices; for an
// "MN-major" operand (instruction-descriptor bit 15 / 16) the rows are K indices and a 16-wide k-step spans two groups.
// Conventions checked on B200 by tools/umma_probe.cu.
__device__ __forceinline__ uint64_t umma_desc_sw(uint32_t smem_addr, uint32_t swizzle_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>(1) << 16;
  d |= static_cast<uint64_t>((8 * swizzle_bytes) >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(swizzle_bytes == 128 ? 2 : 4) << 61;   // 2 = SWIZZLE_128B, 4 = SWIZZLE_64B
  return d;
}
constexpr uint32_t kIdescBMajorMN = 1u << 16;   // B operand is MN-major (rows of the smem tile are K indices)
// kind::f16 instruction descriptor: D=f32 (bit 4), A and B formats in bits 7..9 / 10..12 (0 = fp16, 1 = bf16), both
// K-major, MxN.
__host__ __device__ constexpr uint32_t umma_idesc_f16(int M, int N) {
  return (1u << 4) | (static_cast<uint32_t>(VITED_ACT_BF16) << 7) | (static_cast<uint32_t>(VITED_ACT_BF16) << 10) |
         (static_cast<uint32_t>(N >> 3) << 17) | (static_cast<uint32_t>(M >> 4) << 24);
}

// ---------------------------------------------------------------------------------------------
// legacy warp MMA (used by the small attention tiles only)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void ldsm_x4(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3)
               : "r"(addr));
}
__device__ __forceinline__ void ldsm_x4_trans(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2,
                                              uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3)
               : "r"(addr));
}
__device__ __forceinline__ void mma_f16_16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
#if VITED_ACT_BF16
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, "
#else
      "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, "
#endif
      "{%0, %1, %2, %3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
#endif  // __CUDACC__

}  // namespace vited
