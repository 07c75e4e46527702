// Fused Linear + residual add + LayerNorm for the N = embed_dim = 384 projections of the ViT-ED blocks:
//     x += A * W^T + bias          (attn.proj / cross_attn.proj / mlp.fc2; vision_transformer.py:125-126, :269-271)
//     h  = LayerNorm(x) * g + b    (the NEXT sub-block's norm: norm_cross / norm2 / next layer's norm1; eps 1e-6)
// The unfused path writes the GEMM result as a fp16 `delta`, and a second kernel (resid_ln, 98 % of HBM peak, 23 % of the
// step) re-reads it together with x. Here a CTA pair owns complete 256 x 384 output rows: the accumulator row stays in
// TMEM (384 fp32 columns), the residual tile streams through small TMA boxes, the updated row is parked back in TMEM
// (tcgen05.st) while the row statistics are combined, and the normalised fp16 row leaves through TMA stores.
//
// Structure = gemm_tc_pair_kernel (cta_group::2, TMA ring, one MMA thread) with N = 384 issued as two N = 192 MMAs per
// k-step and a full-row epilogue: 8 epilogue warps per CTA, warp (q, c) owns TMEM lane quarter q (32 rows) and the
// 192-column half c of the row; one thread = one row half. The LayerNorm arithmetic is ln_epilogue.cuh's.
#include "kernels.h"
#include "ln_epilogue.cuh"

namespace vited {

namespace {

constexpr int BM = 128;
constexpr int BK = 64;
constexpr int LN_N = 384;
constexpr int NH = 192;        // columns per MMA

struct LnCfg {
  static constexpr int kEpiWarps = 8;
  static constexpr int kThreads = 128 + 32 * kEpiWarps;
  static constexpr int NW = LN_N / 2;                              // columns per epilogue warp: 192
  static constexpr int XW = 32;                                    // columns per residual box
  static constexpr int CHUNKS = NW / XW;                           // residual boxes per warp and tile: 6
  static constexpr int HW = 64;                                    // columns per pass-2 slab
  static constexpr int SLABS = NW / HW;                            // 3
  static constexpr int ROWB = XW * 4;                              // bytes per box row (= HW * 2) = swizzle span: 128
  static constexpr uint32_t A_BYTES = BM * BK * 2;
  static constexpr uint32_t BH_BYTES = (NH / 2) * BK * 2;          // this CTA's 96 rows of one 192-row weight half
  static constexpr uint32_t STAGE_BYTES = A_BYTES + 2 * BH_BYTES;
  static constexpr int kStages = 3;
  static constexpr uint32_t XBOX = 32 * ROWB;                      // 32 rows x XW fp32, hardware-swizzled: 4 KB
  static constexpr uint32_t X_BYTES = kEpiWarps * 2 * XBOX;        // 64 KB
  static constexpr uint32_t H_BYTES = kEpiWarps * XBOX;            // 32 rows x HW fp16 per warp: 32 KB
  static constexpr uint32_t PARAM_BYTES = 3 * LN_N * 4;
  static constexpr uint32_t PART_BYTES = 2 * BM * 8;                // (mean, M2) of every row half
  static constexpr uint32_t BAR_BYTES = 512;
  static constexpr uint32_t SMEM_BYTES = 1024 + kStages * STAGE_BYTES + X_BYTES + H_BYTES + PARAM_BYTES + PART_BYTES + BAR_BYTES;
  static_assert(SMEM_BYTES <= 232448, "shared memory budget");
  static_assert((2 * kStages + 2 + 2 * kEpiWarps) * 8 + 4 <= BAR_BYTES, "barrier block");
};

#ifdef VITED_LN_TRACE   // clock64 trace of CTA 0 (tools/trace_gemm_ln.py); compiled out of the product library
__device__ unsigned long long g_ln_trace[3 * 32 * 8];   // [0 = epilogue warp (q0,c0), 1 = MMA warp, 2 = epilogue warp (q3,c1)][tile][event]
#define TRL(who, t, ev) do { if (blockIdx.x == 0 && lane == 0 && (t) < 32) g_ln_trace[((who) * 32 + (t)) * 8 + (ev)] = clock64(); } while (0)
#else
#define TRL(who, t, ev) do { } while (0)
#endif

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(LnCfg::kThreads, 1)
gemm_ln_pair_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                    const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmH,
                    const float* __restrict__ bias, const float* __restrict__ ln_w, const float* __restrict__ ln_b,
                    int M, int K, float eps) {
  using Cfg = LnCfg;
  constexpr int kStages = Cfg::kStages;
  constexpr int NW = Cfg::NW, XW = Cfg::XW, CHUNKS = Cfg::CHUNKS, HW = Cfg::HW, ROWB = Cfg::ROWB;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sX = smem + kStages * Cfg::STAGE_BYTES;
  uint8_t* sH = sX + Cfg::X_BYTES;
  float* sBias = reinterpret_cast<float*>(sH + Cfg::H_BYTES);
  float* sG = sBias + LN_N;
  float* sBt = sG + LN_N;
  float2* sPart = reinterpret_cast<float2*>(sBt + LN_N);
  uint64_t* bars = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(sPart) + Cfg::PART_BYTES);
  uint64_t* full = bars;                       // leader CTA: both CTAs' TMA bytes land here
  uint64_t* empty = bars + kStages;            // per CTA, released by the leader's multicast commit
  uint64_t* tfull = bars + 2 * kStages;        // per CTA, multicast commit
  uint64_t* tempty = tfull + 1;                // leader CTA: epilogue warps of BOTH CTAs arrive
  uint64_t* xfull = tempty + 1;                // [8 warps][2 boxes]
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(xfull + 2 * Cfg::kEpiWarps);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int pair = (int)(blockIdx.x >> 1);
  const int num_pairs = (int)(gridDim.x >> 1);
  const int num_tiles = (M + 2 * BM - 1) / (2 * BM);
  const int num_kb = (K + BK - 1) / BK;
  const int my_tiles = pair < num_tiles ? (num_tiles - pair + num_pairs - 1) / num_pairs : 0;

  for (int i = threadIdx.x; i < LN_N; i += Cfg::kThreads) {
    sBias[i] = bias[i];
    sG[i] = ln_w[i];
    sBt[i] = ln_b[i];
  }
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    tma_prefetch_desc(&tmX);
    tma_prefetch_desc(&tmH);
  } else if (warp == 1 && lane == 0) {
    for (int s = 0; s < kStages; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    mbar_init(tfull, 1);
    mbar_init(tempty, 2 * Cfg::kEpiWarps);
    for (int i = 0; i < 2 * Cfg::kEpiWarps; ++i) mbar_init(&xfull[i], 1);
    fence_mbar_init();
  } else if (warp == 2) {
    tmem_alloc_2cta(tmem_holder, 512);
    tmem_relinquish_2cta();
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;

  if (warp == 0) {
    // ===================== TMA producer (both CTAs): own 128 activation rows + 2 x 96 weight rows per k-block ========
    if (lane == 0) {
      uint32_t stage = 0, phase = 0;
      for (int tile = pair; tile < num_tiles; tile += num_pairs) {
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&empty[stage], phase ^ 1, 10);
          uint8_t* a_dst = smem + stage * Cfg::STAGE_BYTES;
          if (rank == 0) mbar_arrive_expect_tx(&full[stage], 2 * Cfg::STAGE_BYTES);
          tma_load_2d_2cta(&tmA, &full[stage], a_dst, kb * BK, tile * 2 * BM + (int)rank * BM);
          tma_load_2d_2cta(&tmB, &full[stage], a_dst + Cfg::A_BYTES, kb * BK, (int)rank * (NH / 2));
          tma_load_2d_2cta(&tmB, &full[stage], a_dst + Cfg::A_BYTES + Cfg::BH_BYTES, kb * BK, NH + (int)rank * (NH / 2));
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA only): two N = 192 MMAs per k-step =====================
    if (rank == 0) {   // warp-uniform loop, tcgen05 instructions predicated on one elected lane
      constexpr uint32_t idesc = umma_idesc_f16(2 * BM, NH);
      constexpr uint32_t kStage16 = Cfg::STAGE_BYTES >> 4, kA16 = Cfg::A_BYTES >> 4, kBH16 = Cfg::BH_BYTES >> 4;
      const uint32_t lo0 = umma_desc_sw128_lo(smem_u32(smem));   // stage 0: A tile, then the two 96-row weight halves
      uint32_t stage = 0, phase = 0, aphase = 0;
      int tt = 0; (void)tt;
      for (int tile = pair; tile < num_tiles; tile += num_pairs, ++tt) {
        TRL(1, tt, 0);
        mbar_wait(tempty, aphase ^ 1, 20);
        TRL(1, tt, 1);
        tc_fence_after();
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&full[stage], phase, 21);
          tc_fence_after();
          const uint32_t lo_a = lo0 + stage * kStage16;
          if (elect_one_sync()) {
#pragma unroll
            for (int k = 0; k < BK / 16; ++k) {
              const uint64_t da = umma_desc_pack(lo_a + 2 * k, kUmmaDescSw128Hi);
              umma_f16_2cta(tmem_base, da, umma_desc_pack(lo_a + kA16 + 2 * k, kUmmaDescSw128Hi), idesc,
                             (kb | k) != 0 ? 1u : 0u);
              umma_f16_2cta(tmem_base + NH, da, umma_desc_pack(lo_a + kA16 + kBH16 + 2 * k, kUmmaDescSw128Hi), idesc,
                             (kb | k) != 0 ? 1u : 0u);
            }
            umma_commit_2cta(&empty[stage]);
          }
          __syncwarp();
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
        if (elect_one_sync()) umma_commit_2cta(tfull);
        __syncwarp();
        TRL(1, tt, 2);
        aphase ^= 1;
      }
    }
  } else if (warp >= 4) {
    // ===================== full-row epilogue (both CTAs, own 128 rows) =====================
    const int ew = warp - 4;
    const int q = warp & 3;       // TMEM lane quarter: rows q*32 .. q*32+31 of this CTA's 128
    const int c = ew >> 2;        // row half: columns [c * NW, (c + 1) * NW)
    uint8_t* xbox = sX + ew * 2 * Cfg::XBOX;
    uint8_t* hbox = sH + ew * Cfg::XBOX;
    uint64_t* my_xfull = xfull + ew * 2;
    const int total_chunks = my_tiles * CHUNKS;
    const uint32_t tlane = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + c * NW;
    // residual boxes are prefetched two chunks ahead, across tile boundaries (so the next tile's first boxes are in
    // flight while the tensor core works on it)
    auto issue_x = [&](int g) {   // lane 0 only
      if (g >= total_chunks) return;
      const int t = g / CHUNKS, j = g - t * CHUNKS;
      const int tile = pair + t * num_pairs;
      mbar_arrive_expect_tx(&my_xfull[g & 1], Cfg::XBOX);
      tma_load_2d(&tmX, &my_xfull[g & 1], xbox + (g & 1) * Cfg::XBOX, c * NW + j * XW, tile * 2 * BM + (int)rank * BM + q * 32);
    };
    if (lane == 0) { issue_x(0); issue_x(1); }
    uint32_t aphase = 0;
    int g = 0;
    for (int t = 0; t < my_tiles; ++t) {
      const int tile = pair + t * num_pairs;
      const int row0 = tile * 2 * BM + (int)rank * BM + q * 32;
      const int who = ew == 0 ? 0 : (ew == Cfg::kEpiWarps - 1 ? 2 : -1); (void)who;
      if (who >= 0) TRL(who, t, 0);
      mbar_wait(tfull, aphase, 30);
      if (who >= 0) TRL(who, t, 1);
      tc_fence_after();
      // ---- pass 1: v = acc + bias + x; park v in TMEM, write it back to the residual stream, shifted statistics ----
      float s = 0.f, ss = 0.f, c0 = 0.f;
#pragma unroll 1
      for (int j = 0; j < CHUNKS; ++j, ++g) {
        const int col0 = c * NW + j * XW;
        uint32_t acc[XW];
        tmem_ld_cols(tlane + j * XW, acc);
        mbar_wait(&my_xfull[g & 1], (uint32_t)(g >> 1) & 1u, 31);
        tmem_ld_wait();
        // shared-window addresses of this lane's row in the in-box / out-box (16-byte chunk i lives at swz_chunk(i))
        const uint32_t in_row = smem_u32(xbox) + (uint32_t)(g & 1) * Cfg::XBOX + lane * ROWB;
        const uint32_t out_row = smem_u32(hbox) + lane * ROWB;
        const uint32_t bias_a = smem_u32(sBias) + col0 * 4;
        // the updated row leaves through the warp's staging box (idle during this pass), NOT through the box it
        // came in: the in-box can then be refilled as soon as the warp has read it, without waiting for a store
        if (lane == 0) tma_store_wait_read();     // the previous chunk's store has finished reading the out-box
        __syncwarp();
        // first the updated row: it goes to the out-box at once, so that the stores have drained by the time the proxy
        // fence in front of the TMA store is reached (MEMBAR.ALL.CTA waits for every store in flight: ~300 cycles when it
        // came right behind the last store); the statistics are computed while they drain
#pragma unroll
        for (int i = 0; i < XW / 4; ++i) {
          const uint32_t off = swz_chunk<ROWB>(i, lane) << 4;
          const float4 xv = lds_f4(in_row + off);
          const float4 b4 = lds_f4(bias_a + 16 * i);
          const float4 v = ln_resid4(acc + 4 * i, b4, xv);
          sts_f4(out_row + off, v);
          acc[4 * i + 0] = __float_as_uint(v.x); acc[4 * i + 1] = __float_as_uint(v.y);
          acc[4 * i + 2] = __float_as_uint(v.z); acc[4 * i + 3] = __float_as_uint(v.w);
        }
        if (j == 0) c0 = __uint_as_float(acc[0]);
        ln_accum_stats(acc, c0, s, ss);
        tmem_st_cols(tlane + j * XW, acc);
        fence_proxy_async_smem();
        __syncwarp();                             // every lane has read the in-box and written the out-box
        if (lane == 0) {
          issue_x(g + 2);                         // refill the in-box right away
          tma_store_2d(&tmX, hbox, col0, row0);
          tma_store_commit();
        }
      }
      tmem_st_wait();
      if (who >= 0) TRL(who, t, 2);
      // ---- combine the two row halves (the q-th pair of warps meets at named barrier q + 1) ----
      uint64_t nmean2, rstd2;
      ln_row_stats<NW, 64>(&sPart[c * BM + q * 32 + lane], &sPart[(c ^ 1) * BM + q * 32 + lane], q + 1, s, ss, c0, eps,
                           nmean2, rstd2);
      if (who >= 0) TRL(who, t, 3);
      // ---- pass 2: normalise out of TMEM, fp16, HW-column slabs through the warp's staging box ----
      const uint32_t hbox_a = smem_u32(hbox) + lane * ROWB, g_a = smem_u32(sG), bt_a = smem_u32(sBt);
#pragma unroll 1
      for (int jj = 0; jj < Cfg::SLABS; ++jj) {
        if (lane == 0) tma_store_wait_read();
        __syncwarp();
#pragma unroll
        for (int hh = 0; hh < HW / 32; ++hh) {
          const int j = jj * (HW / 32) + hh;          // 32-column group of this warp's NW columns
          const int col0 = c * NW + j * 32;
          uint32_t v[32];
          tmem_ld_32x32b_x32(tlane + j * 32, v);
          tmem_ld_wait();
          if (j == NW / 32 - 1) {
            // last read of this tile's accumulator: hand TMEM back to the MMA warp
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_leader(tempty);
          }
#pragma unroll
          for (int i = 0; i < 4; ++i)
            sts_u4(hbox_a + (swz_chunk<ROWB>(hh * 4 + i, lane) << 4),
                   ln_normalise8(v + 8 * i, g_a + col0 * 4 + 32 * i, bt_a + col0 * 4 + 32 * i, nmean2, rstd2));
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          tma_store_2d(&tmH, hbox, c * NW + jj * HW, row0);
          tma_store_commit();
        }
      }
      if (who >= 0) TRL(who, t, 4);
      // (the next tile's sPart entries cannot overtake a partner still reading this tile's: they are written after the
      //  next tfull, which needs tempty of this tile, i.e. every epilogue warp's pass 2 -- behind its sPart reads)
      aphase ^= 1;
    }
    if (lane == 0) tma_store_wait_all();
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc_2cta(tmem_base, 512);
  }
}

}  // namespace

bool gemm_resid_ln_supported(int M, int N, int K) { return N == LN_N && K % 8 == 0 && K >= 8 && M >= 1; }

int gemm_resid_ln(const act_t* A, const act_t* W, const float* bias, float* x, const float* ln_w, const float* ln_b,
                  act_t* h, int M, int N, int K, float eps, cudaStream_t stream) {
  VITED_CHECK(gemm_resid_ln_supported(M, N, K), "gemm_resid_ln: unsupported shape M=%d N=%d K=%d (N must be 384)", M, N, K);
  VITED_CHECK(((reinterpret_cast<uintptr_t>(A) | reinterpret_cast<uintptr_t>(W) | reinterpret_cast<uintptr_t>(x) |
                reinterpret_cast<uintptr_t>(h)) & 15) == 0, "gemm_resid_ln: operands must be 16-byte aligned");
  using Cfg = LnCfg;
  const int sms = gemm_num_sms();
  VITED_CHECK(sms >= 2, "gemm_resid_ln: no device");
  static PerDeviceOnce once;
  if (once.first())
    VITED_CUDA_OK(cudaFuncSetAttribute(gemm_ln_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)Cfg::SMEM_BYTES));
  CUtensorMap tA, tB, tX, tH;
  if (make_tmap_act_2d(&tA, A, (uint64_t)K, (uint64_t)M, (uint64_t)K * 2, 64, BM, 128)) return 1;
  if (make_tmap_act_2d(&tB, W, (uint64_t)K, (uint64_t)N, (uint64_t)K * 2, 64, NH / 2, 128)) return 1;
  if (make_tmap_f32_2d(&tX, x, (uint64_t)N, (uint64_t)M, (uint64_t)N * 4, Cfg::XW, 32, Cfg::ROWB)) return 1;
  if (make_tmap_act_2d(&tH, h, (uint64_t)N, (uint64_t)M, (uint64_t)N * 2, Cfg::HW, 32, Cfg::ROWB)) return 1;
  const int tiles = (M + 2 * BM - 1) / (2 * BM);
  int pairs = sms / 2;
  if (pairs > tiles) pairs = tiles;
  gemm_ln_pair_kernel<<<2 * pairs, Cfg::kThreads, Cfg::SMEM_BYTES, stream>>>(tA, tB, tX, tH, bias, ln_w, ln_b, M, K, eps);
  VITED_CUDA_OK(cudaGetLastError());
  return 0;
}

}  // namespace vited

#ifdef VITED_LN_TRACE
extern "C" __attribute__((visibility("default"))) int vited_debug_ln_trace(unsigned long long* out) {
  return (int)cudaMemcpyFromSymbol(out, vited::g_ln_trace, sizeof(unsigned long long) * 3 * 32 * 8);
}
#endif
