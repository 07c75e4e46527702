// Fused MLP sub-block of the ViT-ED blocks in ONE kernel (embed_dim 384):
//     x += fc2(GELU(fc1(h) + b1)) + b2      (timm Mlp inside Block / CrossBlock: vision_transformer.py:126, :272)
//     h  = LayerNorm(x) * g + b              (the NEXT layer's norm1; eps 1e-6)
// The unfused sequence writes the [rows, 1536] hidden activations to HBM (fc1 + GELU epilogue) and reads them back
// (fc2): 6 KB of the 10.7 KB per row those two launches move. Here the hidden activations never leave the SM.
//
// A CTA pair owns complete 256 x 384 output rows (cta_group::2, 128 rows per CTA). Per tile:
//   * the h tile (A operand of fc1, 128 x 384 fp16 per CTA = 96 KB) is loaded ONCE and stays in shared memory;
//   * the hidden dimension is walked in chunks of 64: S_c = h W1_c^T (M 256, N 64, K 384) into one of two 64-column
//     TMEM buffers; the eight GELU warps turn S_c + b1 into fp16 probabilities-style operands P_c written back over S_c
//     (tcgen05.st, packed pairs) and the second MMA takes P_c as its A operand straight from TMEM:
//     O += P_c W2_c^T (M 256, N 2 x 192, K 64) into the 384-column output accumulator;
//   * issue order G1(0) G1(1) | G2(c) G1(c+2) ...: the tensor pipe runs fc1 of chunk c+1 while the GELU warps work on
//     chunk c; the weight chunks (W1_c: 64 x 384, W2_c: 384 x 64) stream from L2 through a ring of 12-KB slots;
//   * the full-row epilogue of gemm_ln.cu (residual tile through TMA boxes, updated row parked in TMEM, shifted one-pass
//     statistics, Chan combination of the two column halves, normalise, TMA stores) runs on the same eight warps. Its
//     residual boxes live in the h-tile region, which is dead once fc1 of the last chunk has completed.
// TMEM: O = columns [0, 384), S buffers [384, 448) and [448, 512). Shared memory: 96 KB h tile / residual boxes,
// 96 KB weight ring, 16 KB output staging, biases / LayerNorm parameters.
// Template parameter CG = column groups of the GELU / epilogue warps: 2 (8 warps: 32 hidden columns of a chunk and a
// 192-column half row each) or 4 (16 warps: 16 hidden columns and a 96-column quarter row each, residual boxes of half
// the width, weight ring of 6 slots, 32 KB staging) -- same bytes, twice as many independent chains in flight.
//
// Template parameter PRO adds the cross-attention projection in front (cproj_mlp_resid_ln, the decoder's
//     x_mid = x + o W_cproj^T + b_cproj;  h = norm2(x_mid);  then the MLP sub-block above on h and x_mid):
//   * the h-tile producer loads the `o` tile into the h-tile region; the weight producer streams W_cproj ahead of
//     W1 / W2 (one 12-KB slot = this CTA's 96 rows of an N half x one 64-column k-block, 12 slots per tile);
//   * the issuer runs O = o W_cproj^T into TMEM columns [0, 384) (6 k-blocks x 2 N halves) and commits proj_done;
//   * prologue pass 1 (gemm_ln.cu's arithmetic, operation for operation): x_mid = O + (b_cproj + x) with x through the
//     residual boxes in the now dead h-tile region, shifted statistics, 2 x_mid parked in the same TMEM columns;
//   * prologue pass 2 normalises 0.5 * park (exact) with norm2 and writes h as 16-bit values straight into the h-tile
//     region in the 128B-swizzled K-major layout fc1's descriptor reads (h is bit-identical to gemm_ln's);
//   * fc2 accumulates onto the parked 2 x_mid (the hidden operands are 2 GELU), so the epilogue's v = 0.5 O + b2 needs
//     no residual read: x_mid and h never reach global memory.
#include "kernels.h"

namespace vited {

namespace {

constexpr int BM = 128;
constexpr int BK = 64;
constexpr int LN_N = 384;
constexpr int NH = 192;          // columns per fc2 MMA
constexpr int HC = 64;           // hidden units per chunk
constexpr int KB1 = LN_N / BK;   // k-blocks of fc1 (K = 384)

template <int CG>
struct MlpCfg {
  static_assert(CG == 2 || CG == 4, "two or four column groups");
  static constexpr int kEpiWarps = 4 * CG;
  static constexpr int kThreads = 128 + 32 * kEpiWarps;
  static constexpr int NW = LN_N / CG;                                // output columns per epilogue warp: 192 / 96
  static constexpr int XW = 64 / CG;                                  // columns per residual box: 32 / 16
  static constexpr int CHUNKS = NW / XW;                              // residual boxes per warp and tile: 6
  static constexpr int ROWB = XW * 4;                                 // bytes per residual-box row = swizzle span: 128 / 64
  static constexpr int GW = HC / CG;                                  // hidden columns of a chunk per GELU warp: 32 / 16
  static constexpr uint32_t A_KB_BYTES = BM * BK * 2;                 // one k-block of the h tile: 128 rows x 128 B
  static constexpr uint32_t A_BYTES = KB1 * A_KB_BYTES;               // 96 KB
  static constexpr uint32_t SLOT_BYTES = 12288;                       // 3 k-blocks of W1 (32 rows each) or 96 rows of W2
  // 6 slots left the issuer waiting for weights 11.6 k of 63 k cycles per tile (trace), 8 changed nothing in the step:
  // the issuer runs ahead of the tensor pipe by the ring depth. The 16-warp form needs the 24 KB for its staging boxes.
  static constexpr int kSlots = CG == 2 ? 8 : 6;
  static constexpr uint32_t W1_KB_BYTES = (HC / 2) * BK * 2;          // this CTA's 32 rows of one k-block: 4 KB
  static constexpr uint32_t XBOX = 32 * ROWB;                         // 32 rows x XW fp32, hardware-swizzled: 4 KB / 2 KB
  static constexpr uint32_t OUT_BYTES = kEpiWarps * 2048;             // pass-2 staging: 32 rows x 32 fp16 per warp (64B swizzle)
  static constexpr uint32_t PART_BYTES = CG * BM * 8;                 // (mean, M2) of every row part
  static constexpr uint32_t BAR_BYTES = 512;
  static_assert(kEpiWarps * 3 * XBOX == A_BYTES, "the residual boxes (2 in + 1 out per warp) reuse the h-tile region");
  static_assert((2 * kSlots + 9 + 2 * kEpiWarps + 3) * 8 <= BAR_BYTES, "barrier block");
  static uint32_t smem_bytes(int hidden, bool pro) {   // pro: + b_cproj and the norm2 parameters
    return 1024 + A_BYTES + kSlots * SLOT_BYTES + OUT_BYTES + (uint32_t)hidden * 4 + (pro ? 6 : 3) * LN_N * 4 + PART_BYTES +
           BAR_BYTES;
  }
};

constexpr uint32_t kColS = LN_N;   // first TMEM column of the two hidden-chunk buffers

#ifdef VITED_MLP_TRACE   // clock64 trace of CTA 0 (tools/trace_mlp_ln.py); compiled out of the product library
__device__ long long g_mlp_trace[2 * 32 * 8];   // [0 = GELU/epilogue warp (q0,c0), 1 = MMA warp][tile][event]
#define TRM(who, t, ev, val) do { if (blockIdx.x == 0 && lane == 0 && (t) < 32) g_mlp_trace[((who) * 32 + (t)) * 8 + (ev)] = (val); } while (0)
#define TRM_CLK() clock64()
__device__ long long g_mlp_trace2[32 * 8];      // pass-1 breakdown of epilogue warp (q0, c0) per tile, summed over its chunks
#define TR2(t, ev, val) do { if (blockIdx.x == 0 && ew == 0 && lane == 0 && (t) < 32) g_mlp_trace2[(t) * 8 + (ev)] = (val); } while (0)
#define TR2_ACC(accu, c0, c1) do { accu += (c1) - (c0); } while (0)
#else
#define TR2(t, ev, val) do { } while (0)
#define TR2_ACC(accu, c0, c1) do { } while (0)
#define TRM(who, t, ev, val) do { } while (0)
#define TRM_CLK() 0ll
#endif

template <int CG, bool PRO>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(MlpCfg<CG>::kThreads, 1)
mlp_ln_pair_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmWp,
                   const __grid_constant__ CUtensorMap tmW1, const __grid_constant__ CUtensorMap tmW2,
                   const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmH,
                   const float* __restrict__ bproj, const float* __restrict__ ln2_w, const float* __restrict__ ln2_b,
                   const float* __restrict__ b1, const float* __restrict__ b2, const float* __restrict__ ln_w,
                   const float* __restrict__ ln_b, int M, int hidden, float eps) {
  using Cfg = MlpCfg<CG>;
  constexpr int kSlots = Cfg::kSlots;
  constexpr int NW = Cfg::NW, XW = Cfg::XW, CHUNKS = Cfg::CHUNKS, ROWB = Cfg::ROWB, GW = Cfg::GW;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sA = smem;                                  // h tile (PRO: first the o tile); residual boxes in the epilogues
  uint8_t* sW = sA + Cfg::A_BYTES;                     // weight ring
  uint8_t* sOut = sW + kSlots * Cfg::SLOT_BYTES;       // pass-2 staging
  float* sB1 = reinterpret_cast<float*>(sOut + Cfg::OUT_BYTES);
  float* sBias = sB1 + hidden;
  float* sG = sBias + LN_N;
  float* sBt = sG + LN_N;
  float* sBp = sBt + LN_N;                             // PRO: b_cproj, norm2 weight and bias
  float* sG2 = sBp + LN_N;
  float* sBt2 = sG2 + LN_N;
  float2* sPart = reinterpret_cast<float2*>(PRO ? sBt2 + LN_N : sBp);
  uint64_t* bars = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(sPart) + Cfg::PART_BYTES);
  uint64_t* w_full = bars;                    // [kSlots] leader CTA: both CTAs' TMA bytes land here
  uint64_t* w_empty = w_full + kSlots;        // [kSlots] per CTA, released by the leader's multicast commit
  uint64_t* a_full = w_empty + kSlots;        // leader CTA: h tile of both CTAs landed
  uint64_t* a_free = a_full + 1;              // per CTA: the 8 local epilogue warps are done with the residual boxes
  uint64_t* s_full = a_free + 1;              // [2] per CTA (multicast commit): S_c complete
  uint64_t* p_full = s_full + 2;              // [2] leader CTA: the GELU warps of BOTH CTAs have written P_c
  uint64_t* g1_done = p_full + 2;             // per CTA (multicast commit): fc1 of the tile's last chunk has read the h tile
  uint64_t* tfull = g1_done + 1;              // per CTA (multicast commit): O complete
  uint64_t* tempty = tfull + 1;               // leader CTA: epilogue warps of BOTH CTAs have drained O
  uint64_t* xfull = tempty + 1;               // [epilogue warps][2 boxes]
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(xfull + 2 * Cfg::kEpiWarps);
  uint64_t* proj_done = xfull + 2 * Cfg::kEpiWarps + 1;   // PRO, per CTA (multicast commit): O = o W_cproj^T complete
  uint64_t* h_full = proj_done + 1;           // PRO, leader CTA: the epilogue warps of BOTH CTAs have written their h
                                              // tile and are done with the park (written and read)

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int pair = (int)(blockIdx.x >> 1);
  const int num_pairs = (int)(gridDim.x >> 1);
  const int num_tiles = (M + 2 * BM - 1) / (2 * BM);
  const int n_chunks = hidden / HC;
  const int my_tiles = pair < num_tiles ? (num_tiles - pair + num_pairs - 1) / num_pairs : 0;

  for (int i = threadIdx.x; i < hidden; i += Cfg::kThreads) sB1[i] = b1[i];
  for (int i = threadIdx.x; i < LN_N; i += Cfg::kThreads) {
    sBias[i] = b2[i];
    sG[i] = ln_w[i];
    sBt[i] = ln_b[i];
    if constexpr (PRO) {
      sBp[i] = bproj[i];
      sG2[i] = ln2_w[i];
      sBt2[i] = ln2_b[i];
    }
  }
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    if constexpr (PRO) tma_prefetch_desc(&tmWp);
    tma_prefetch_desc(&tmW1);
    tma_prefetch_desc(&tmW2);
    tma_prefetch_desc(&tmX);
    tma_prefetch_desc(&tmH);
  } else if (warp == 1 && lane == 0) {
    for (int s = 0; s < kSlots; ++s) {
      mbar_init(&w_full[s], 1);
      mbar_init(&w_empty[s], 1);
    }
    mbar_init(a_full, 1);
    mbar_init(a_free, Cfg::kEpiWarps);
    for (int s = 0; s < 2; ++s) {
      mbar_init(&s_full[s], 1);
      mbar_init(&p_full[s], 2 * Cfg::kEpiWarps);
    }
    mbar_init(g1_done, 1);
    mbar_init(tfull, 1);
    mbar_init(tempty, 2 * Cfg::kEpiWarps);
    for (int i = 0; i < 2 * Cfg::kEpiWarps; ++i) mbar_init(&xfull[i], 1);
    if constexpr (PRO) {
      mbar_init(proj_done, 1);
      mbar_init(h_full, 2 * Cfg::kEpiWarps);
    }
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
  pdl_launch_dependents();
  pdl_wait();           // the prologue above overlapped the previous kernel's tail; global memory only from here on

  if (warp == 0) {
    // ===================== weight producer (both CTAs): slots in the order the issuer consumes them ================
    // step sequence of a tile: G1(0) G1(1) | G2(0) G1(2) | G2(1) G1(3) | ... | G2(n-3) G1(n-1) | G2(n-2) G2(n-1);
    // every step takes two slots (fc1: k-blocks 0-2 / 3-5 of this CTA's 32 rows; fc2: this CTA's 96 rows of each N half)
    if (lane == 0) {
      uint32_t slot = 0, phase = 0;
      auto load_w1 = [&](int c) {
        for (int hf = 0; hf < 2; ++hf) {
          mbar_wait(&w_empty[slot], phase ^ 1, 10);
          uint8_t* dst = sW + slot * Cfg::SLOT_BYTES;
          if (rank == 0) mbar_arrive_expect_tx(&w_full[slot], 2 * Cfg::SLOT_BYTES);
          for (int j = 0; j < 3; ++j)
            tma_load_2d_2cta(&tmW1, &w_full[slot], dst + j * Cfg::W1_KB_BYTES, (hf * 3 + j) * BK, c * HC + (int)rank * (HC / 2));
          if (++slot == kSlots) { slot = 0; phase ^= 1; }
        }
      };
      auto load_w2 = [&](int c) {
        for (int hf = 0; hf < 2; ++hf) {
          mbar_wait(&w_empty[slot], phase ^ 1, 11);
          uint8_t* dst = sW + slot * Cfg::SLOT_BYTES;
          if (rank == 0) mbar_arrive_expect_tx(&w_full[slot], 2 * Cfg::SLOT_BYTES);
          tma_load_2d_2cta(&tmW2, &w_full[slot], dst, c * HC, hf * NH + (int)rank * (NH / 2));
          if (++slot == kSlots) { slot = 0; phase ^= 1; }
        }
      };
      auto load_wp = [&]() {   // W_cproj: k-block kb of this CTA's 96 rows of N half hf per slot
        for (int kb = 0; kb < KB1; ++kb)
          for (int hf = 0; hf < 2; ++hf) {
            mbar_wait(&w_empty[slot], phase ^ 1, 13);
            uint8_t* dst = sW + slot * Cfg::SLOT_BYTES;
            if (rank == 0) mbar_arrive_expect_tx(&w_full[slot], 2 * Cfg::SLOT_BYTES);
            tma_load_2d_2cta(&tmWp, &w_full[slot], dst, kb * BK, hf * NH + (int)rank * (NH / 2));
            if (++slot == kSlots) { slot = 0; phase ^= 1; }
          }
      };
      for (int t = 0; t < my_tiles; ++t) {
        if constexpr (PRO) load_wp();
        load_w1(0);
        if (n_chunks > 1) load_w1(1);
        for (int c = 0; c < n_chunks; ++c) {
          load_w2(c);
          if (c + 2 < n_chunks) load_w1(c + 2);
        }
      }
    }
  } else if (warp == 3) {
    // ===================== h-tile producer (both CTAs; PRO: the o tile): own 128 rows, all six k-blocks =============
    if (lane == 0) {
      for (int t = 0; t < my_tiles; ++t) {
        const int tile = pair + t * num_pairs;
        // (an L2 prefetch of these rows issued at g1_done of the previous tile -- a whole epilogue ahead of the load --
        //  measured 0.5470 vs 0.5455 ms: no gain; profiles/README.md item 43)
        mbar_wait(a_free, (uint32_t)(t & 1) ^ 1u, 12);     // the previous tile's residual boxes are done with the region
        if (rank == 0) mbar_arrive_expect_tx(a_full, 2 * Cfg::A_BYTES);
        for (int kb = 0; kb < KB1; ++kb)
          tma_load_2d_2cta(&tmA, a_full, sA + kb * Cfg::A_KB_BYTES, kb * BK, tile * 2 * BM + (int)rank * BM);
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA only; warp-uniform, tcgen05 on one elected lane) =====================
    if (rank == 0) {
      constexpr uint32_t idesc1 = umma_idesc_f16(2 * BM, HC);
      constexpr uint32_t idesc2 = umma_idesc_f16(2 * BM, NH);
      const uint32_t lo_a0 = umma_desc_sw128_lo(smem_u32(sA));
      const uint32_t lo_w0 = umma_desc_sw128_lo(smem_u32(sW));
      uint32_t slot = 0, phase = 0;
      uint32_t pfull_ph = 0;                               // bit b: parity of the next p_full[b] phase
#ifdef VITED_MLP_TRACE
      long long acc_wait_p = 0, acc_wait_w = 0;
#define TRM_WAIT(accu, stmt) do { const long long _c0 = clock64(); stmt; accu += clock64() - _c0; } while (0)
#else
#define TRM_WAIT(accu, stmt) do { stmt; } while (0)
#endif
      auto g1 = [&](int c, bool last) {                    // S[c & 1] = h W1_c^T
        const uint32_t d_tmem = tmem_base + kColS + (uint32_t)(c & 1) * HC;
        for (int hf = 0; hf < 2; ++hf) {
          TRM_WAIT(acc_wait_w, mbar_wait(&w_full[slot], phase, 21));
          tc_fence_after();
          const uint32_t lo_w = lo_w0 + slot * (Cfg::SLOT_BYTES >> 4);
          if (elect_one_sync()) {
#pragma unroll
            for (int j = 0; j < 3; ++j) {
              const uint32_t lo_a = lo_a0 + (uint32_t)(hf * 3 + j) * (Cfg::A_KB_BYTES >> 4);
#pragma unroll
              for (int k = 0; k < BK / 16; ++k)
                umma_f16_2cta(d_tmem, umma_desc_pack(lo_a + 2 * k, kUmmaDescSw128Hi),
                               umma_desc_pack(lo_w + j * (Cfg::W1_KB_BYTES >> 4) + 2 * k, kUmmaDescSw128Hi), idesc1,
                               (hf | j | k) != 0 ? 1u : 0u);
            }
            umma_commit_2cta(&w_empty[slot]);
          }
          __syncwarp();
          if (++slot == kSlots) { slot = 0; phase ^= 1; }
        }
        if (elect_one_sync()) {
          umma_commit_2cta(&s_full[c & 1]);
          if (last) umma_commit_2cta(g1_done);
        }
        __syncwarp();
      };
      auto g2 = [&](int c, bool last) {                    // O += P_c W2_c^T, P_c from TMEM
        const int b = c & 1;
        TRM_WAIT(acc_wait_p, mbar_wait(&p_full[b], (pfull_ph >> b) & 1u, 22));
        pfull_ph ^= 1u << b;
        tc_fence_after();
        // P_c: GELU column group g (GW hidden units) leaves its GW / 2 packed columns at S + g * GW, so the 16 hidden
        // units of k-step k start at column (16k / GW) * GW + (16k % GW) / 2
        const uint32_t a_tmem = tmem_base + kColS + (uint32_t)b * HC;
        for (int hf = 0; hf < 2; ++hf) {
          TRM_WAIT(acc_wait_w, mbar_wait(&w_full[slot], phase, 23));
          tc_fence_after();
          const uint32_t lo_w = lo_w0 + slot * (Cfg::SLOT_BYTES >> 4);
          if (elect_one_sync()) {
#pragma unroll
            for (int k = 0; k < HC / 16; ++k)
              umma_f16_ts_2cta(tmem_base + hf * NH, a_tmem + (uint32_t)((16 * k / GW) * GW + (16 * k % GW) / 2),
                                umma_desc_pack(lo_w + 2 * k, kUmmaDescSw128Hi), idesc2,
                                (PRO || (c | k) != 0) ? 1u : 0u);   // PRO: onto the parked 2 x_mid
            umma_commit_2cta(&w_empty[slot]);
          }
          __syncwarp();
          if (++slot == kSlots) { slot = 0; phase ^= 1; }
        }
        if (last) {
          if (elect_one_sync()) umma_commit_2cta(tfull);
          __syncwarp();
        }
      };
      auto proj = [&]() {                                  // O = o W_cproj^T (k-blocks of the o tile in order, as gemm_ln)
        for (int kb = 0; kb < KB1; ++kb) {
          const uint32_t lo_a = lo_a0 + (uint32_t)kb * (Cfg::A_KB_BYTES >> 4);
          for (int hf = 0; hf < 2; ++hf) {
            mbar_wait(&w_full[slot], phase, 25);
            tc_fence_after();
            const uint32_t lo_w = lo_w0 + slot * (Cfg::SLOT_BYTES >> 4);
            if (elect_one_sync()) {
#pragma unroll
              for (int k = 0; k < BK / 16; ++k)
                umma_f16_2cta(tmem_base + hf * NH, umma_desc_pack(lo_a + 2 * k, kUmmaDescSw128Hi),
                               umma_desc_pack(lo_w + 2 * k, kUmmaDescSw128Hi), idesc2, (kb | k) != 0 ? 1u : 0u);
              umma_commit_2cta(&w_empty[slot]);
            }
            __syncwarp();
            if (++slot == kSlots) { slot = 0; phase ^= 1; }
          }
        }
        if (elect_one_sync()) umma_commit_2cta(proj_done);
        __syncwarp();
      };
      for (int t = 0; t < my_tiles; ++t) {
        TRM(1, t, 0, TRM_CLK());
        mbar_wait(a_full, (uint32_t)(t & 1), 20);
        TRM(1, t, 1, TRM_CLK());
        tc_fence_after();
        if constexpr (PRO) {
          mbar_wait(tempty, (uint32_t)(t & 1) ^ 1u, 24);   // the previous tile's epilogue has drained O
          tc_fence_after();
          proj();
          mbar_wait(h_full, (uint32_t)(t & 1), 26);        // both h tiles written; the park is complete and read
          tc_fence_after();
        }
        g1(0, n_chunks == 1);
        if (n_chunks > 1) g1(1, n_chunks == 2);
        for (int c = 0; c < n_chunks; ++c) {
          if (!PRO && c == 0) {                            // the previous tile's epilogue has drained O
            TRM(1, t, 2, TRM_CLK());
            mbar_wait(tempty, (uint32_t)(t & 1) ^ 1u, 24);
            TRM(1, t, 3, TRM_CLK());
            tc_fence_after();
          }
          g2(c, c == n_chunks - 1);
          if (c + 2 < n_chunks) g1(c + 2, c + 3 == n_chunks);
        }
        TRM(1, t, 4, TRM_CLK());
#ifdef VITED_MLP_TRACE
        TRM(1, t, 5, acc_wait_p);
        TRM(1, t, 6, acc_wait_w);
#endif
      }
    }
  } else if (warp >= 4) {
    // ===================== (PRO: cross-proj prologue,) GELU of the hidden chunks, then the full-row epilogue ==========
    // (both CTAs, own 128 rows)
    const int ew = warp - 4;
    const int q = warp & 3;       // TMEM lane quarter: rows q*32 .. q*32+31 of this CTA's 128
    const int c = ew >> 2;        // column group (of a hidden chunk: GW of 64; of the output row: NW of 384)
    uint8_t* xbox = sA + ew * 3 * Cfg::XBOX;             // two in-boxes, then the out-box
    uint8_t* obox = xbox + 2 * Cfg::XBOX;
    uint8_t* hbox = sOut + ew * 2048;
    uint64_t* my_xfull = xfull + ew * 2;
    const uint32_t lane_off = static_cast<uint32_t>(q * 32) << 16;
    const uint32_t tlane = tmem_base + lane_off + c * NW;
    const uint32_t tS = tmem_base + lane_off + kColS + c * GW;
    uint32_t sfull_ph = 0;        // bit b: parity of the next s_full[b] phase
    int g = 0;                    // residual boxes issued / consumed so far (2-deep per warp)
    // shifted one-pass statistics of one chunk of this lane's row part (pivot c0 = the part's first element)
    auto accum_stats = [&](const uint32_t (&acc)[XW], float c0, float& s, float& ss) {
      uint64_t s2[2] = {0ull, 0ull}, q2[2] = {0ull, 0ull};                 // four independent chains each
      const uint64_t nc0 = f2_dup(-c0);
#pragma unroll
      for (int i = 0; i < XW / 2; ++i) {
        const uint64_t d = f2_add(f2_from_bits(acc[2 * i], acc[2 * i + 1]), nc0);
        s2[i & 1] = f2_add(s2[i & 1], d);
        q2[i & 1] = f2_fma(d, d, q2[i & 1]);
      }
      float s4[4], q4[4];
      f2_unpack(s2[0], s4[0], s4[1]); f2_unpack(s2[1], s4[2], s4[3]);
      f2_unpack(q2[0], q4[0], q4[1]); f2_unpack(q2[1], q4[2], q4[3]);
      s += (s4[0] + s4[1]) + (s4[2] + s4[3]);
      ss += (q4[0] + q4[1]) + (q4[2] + q4[3]);
    };
    // combine the CG column groups of every row (Chan): n = NW each. all_warps: exchange over every epilogue warp of
    // the CTA (the prologue: afterwards no warp reads its residual boxes any more) instead of the CG warps of quarter q
    auto row_stats = [&](float s, float ss, float c0, bool all_warps, uint64_t& nmean2, uint64_t& rstd2) {
      const float inv_n = 1.f / NW;
      const float mean_a = c0 + s * inv_n, m2_a = ss - s * s * inv_n;
      sPart[c * BM + q * 32 + lane] = make_float2(mean_a, m2_a);
      if (all_warps) asm volatile("bar.sync 5, %0;" ::"n"(32 * Cfg::kEpiWarps) : "memory");
      else asm volatile("bar.sync %0, %1;" ::"r"(q + 1), "n"(32 * CG) : "memory");
      float mean, var;
      if constexpr (CG == 2) {
        const float2 o = sPart[(c ^ 1) * BM + q * 32 + lane];
        const float dm = o.x - mean_a;
        mean = 0.5f * (mean_a + o.x);
        var = (m2_a + o.y + dm * dm * (0.5f * NW)) * (1.f / LN_N);
      } else {
        float mg[CG], m2 = 0.f, msum = 0.f;
#pragma unroll
        for (int k = 0; k < CG; ++k) {
          const float2 o = sPart[k * BM + q * 32 + lane];
          mg[k] = o.x;
          m2 += o.y;
          msum += o.x;
        }
        mean = msum * (1.f / CG);
        float between = 0.f;
#pragma unroll
        for (int k = 0; k < CG; ++k) between = fmaf(mg[k] - mean, mg[k] - mean, between);
        var = (m2 + between * (float)NW) * (1.f / LN_N);
      }
      const float rstd = rsqrtf(fmaxf(var, 0.f) + eps);
      nmean2 = f2_dup(-mean);
      rstd2 = f2_dup(rstd);
    };
    // 8 normalised 16-bit values of columns [col, col + 8) (g_a / bt_a: shared-window address of column col's parameters)
    auto normalise8 = [&](const uint32_t* v, uint32_t g_a, uint32_t bt_a, uint64_t nmean2, uint64_t rstd2) {
      const float4 g0 = lds_f4(g_a);
      const float4 g1v = lds_f4(g_a + 16);
      const float4 t0 = lds_f4(bt_a);
      const float4 t1 = lds_f4(bt_a + 16);
      float y[8];
      f2_unpack(f2_fma(f2_mul(f2_add(f2_from_bits(v[0], v[1]), nmean2), rstd2), f2_pack(g0.x, g0.y), f2_pack(t0.x, t0.y)), y[0], y[1]);
      f2_unpack(f2_fma(f2_mul(f2_add(f2_from_bits(v[2], v[3]), nmean2), rstd2), f2_pack(g0.z, g0.w), f2_pack(t0.z, t0.w)), y[2], y[3]);
      f2_unpack(f2_fma(f2_mul(f2_add(f2_from_bits(v[4], v[5]), nmean2), rstd2), f2_pack(g1v.x, g1v.y), f2_pack(t1.x, t1.y)), y[4], y[5]);
      f2_unpack(f2_fma(f2_mul(f2_add(f2_from_bits(v[6], v[7]), nmean2), rstd2), f2_pack(g1v.z, g1v.w), f2_pack(t1.z, t1.w)), y[6], y[7]);
      uint4 pk;
      pk.x = pack_act(y[0], y[1]);
      pk.y = pack_act(y[2], y[3]);
      pk.z = pack_act(y[4], y[5]);
      pk.w = pack_act(y[6], y[7]);
      return pk;
    };
    for (int t = 0; t < my_tiles; ++t) {
      const int tile = pair + t * num_pairs;
      const int row0 = tile * 2 * BM + (int)rank * BM + q * 32;
      auto issue_x = [&](int j, int gg) {   // lane 0 only: 32-row x XW-column fp32 box j of this warp's row part
        mbar_arrive_expect_tx(&my_xfull[gg & 1], Cfg::XBOX);
        tma_load_2d(&tmX, &my_xfull[gg & 1], xbox + (gg & 1) * Cfg::XBOX, c * NW + j * XW, row0);
      };
      if constexpr (PRO) {
        // ---- prologue pass 1: x_mid = O + (b_cproj + x), shifted statistics; 2 x_mid parked in TMEM, not stored.
        //      The o tile is dead once the projection has completed: its region takes the residual boxes ----
        mbar_wait(proj_done, (uint32_t)(t & 1), 34);
        if (lane == 0) {
          issue_x(0, g);
          issue_x(1, g + 1);
        }
        tc_fence_after();
        float s = 0.f, ss = 0.f, c0 = 0.f;
#pragma unroll 1
        for (int j = 0; j < CHUNKS; ++j, ++g) {
          uint32_t acc[XW];
          tmem_ld_cols(tlane + j * XW, acc);
          mbar_wait(&my_xfull[g & 1], (uint32_t)(g >> 1) & 1u, 35);
          tmem_ld_wait();
          const uint32_t in_row = smem_u32(xbox) + (uint32_t)(g & 1) * Cfg::XBOX + lane * ROWB;
          const uint32_t bias_a = smem_u32(sBp) + (c * NW + j * XW) * 4;
#pragma unroll
          for (int i = 0; i < XW / 4; ++i) {
            const float4 xv = lds_f4(in_row + (swz_chunk<ROWB>(i, lane) << 4));
            const float4 b4 = lds_f4(bias_a + 16 * i);
            float4 v;
            f2_unpack(f2_add(f2_from_bits(acc[4 * i + 0], acc[4 * i + 1]), f2_add(f2_pack(b4.x, b4.y), f2_pack(xv.x, xv.y))), v.x, v.y);
            f2_unpack(f2_add(f2_from_bits(acc[4 * i + 2], acc[4 * i + 3]), f2_add(f2_pack(b4.z, b4.w), f2_pack(xv.z, xv.w))), v.z, v.w);
            acc[4 * i + 0] = __float_as_uint(v.x); acc[4 * i + 1] = __float_as_uint(v.y);
            acc[4 * i + 2] = __float_as_uint(v.z); acc[4 * i + 3] = __float_as_uint(v.w);
          }
          __syncwarp();                           // every lane has read the in-box: refill it
          if (lane == 0 && j + 2 < CHUNKS) issue_x(j + 2, g + 2);
          if (j == 0) c0 = __uint_as_float(acc[0]);
          accum_stats(acc, c0, s, ss);
#pragma unroll
          for (int i = 0; i < XW / 2; ++i) {      // park 2 x_mid (exact): fc2 accumulates onto it
            float lo, hi;
            f2_unpack(f2_mul(f2_from_bits(acc[2 * i], acc[2 * i + 1]), f2_dup(2.f)), lo, hi);
            acc[2 * i] = __float_as_uint(lo);
            acc[2 * i + 1] = __float_as_uint(hi);
          }
          tmem_st_cols(tlane + j * XW, acc);
        }
        tmem_st_wait();
        uint64_t nmean2, rstd2;
        row_stats(s, ss, c0, true, nmean2, rstd2);
        // ---- prologue pass 2: h = norm2(0.5 park) as 16-bit values straight into the h tile: row r of k-block kb at
        //      kb * 16 KB + r * 128 B, 16-byte chunk i at i ^ (r & 7) (the 128B swizzle fc1's descriptor reads) ----
        const uint32_t h_row = smem_u32(sA) + (uint32_t)(q * 32 + lane) * 128;
#pragma unroll 1
        for (int j = 0; j < NW / 32; ++j) {
          const int col0 = c * NW + j * 32;
          uint32_t v[32];
          tmem_ld_32x32b_x32(tlane + j * 32, v);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            float lo, hi;
            f2_unpack(f2_mul(f2_from_bits(v[2 * i], v[2 * i + 1]), f2_dup(0.5f)), lo, hi);
            v[2 * i] = __float_as_uint(lo);
            v[2 * i + 1] = __float_as_uint(hi);
          }
          const uint32_t dst = h_row + (uint32_t)(col0 / BK) * Cfg::A_KB_BYTES;
#pragma unroll
          for (int i = 0; i < 4; ++i)
            sts_u4(dst + (swz_chunk<128>((col0 % BK) / 8 + i, lane) << 4),
                   normalise8(v + 8 * i, smem_u32(sG2) + (col0 + 8 * i) * 4, smem_u32(sBt2) + (col0 + 8 * i) * 4, nmean2,
                              rstd2));
        }
        fence_proxy_async_smem();                 // the h tile is read by the tensor core (async proxy)
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_leader(h_full);
      }
      // ---- GELU: P_c = gelu(S_c + b1) as packed fp16 pairs over the first half of this warp's GW S columns ----
#ifdef VITED_MLP_TRACE
      long long acc_wait_s = 0;
      if (ew == 0) TRM(0, t, 0, TRM_CLK());
#endif
      for (int ch = 0; ch < n_chunks; ++ch) {
        const int b = ch & 1;
        TRM_WAIT(acc_wait_s, mbar_wait(&s_full[b], (sfull_ph >> b) & 1u, 32));
        sfull_ph ^= 1u << b;
        tc_fence_after();
        uint32_t acc[GW];
        tmem_ld_cols(tS + b * HC, acc);
        tmem_ld_wait();
        const uint32_t bp = smem_u32(sB1) + (uint32_t)(ch * HC + c * GW) * 4;
        uint32_t pk[GW / 2];
#pragma unroll
        for (int i = 0; i < GW / 4; ++i) {
          // P_c holds TWICE the GELU (gelu2x_fast2: 4.5 instead of 8.5 issue slots per element; GELU(c) sits between
          // fc1(c + 1) and fc2(c) on the tensor pipe's critical path); pass 1 of the epilogue halves the accumulator
          const float4 b4 = lds_f4(bp + 16 * i);
          float v0, v1, v2, v3;
          f2_unpack(gelu2x_fast2(f2_add(f2_from_bits(acc[4 * i + 0], acc[4 * i + 1]), f2_pack(b4.x, b4.y))), v0, v1);
          f2_unpack(gelu2x_fast2(f2_add(f2_from_bits(acc[4 * i + 2], acc[4 * i + 3]), f2_pack(b4.z, b4.w))), v2, v3);
          pk[2 * i] = pack_act(v0, v1);
          pk[2 * i + 1] = pack_act(v2, v3);
        }
        tmem_st_cols(tS + b * HC, pk);
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_leader(&p_full[b]);
      }
      // ---- the h tile is dead once fc1 of the last chunk has completed: its region now takes the residual boxes ----
#ifdef VITED_MLP_TRACE
      if (ew == 0) { TRM(0, t, 1, TRM_CLK()); TRM(0, t, 6, acc_wait_s); }
#endif
      if (lane == 0) {
        mbar_wait(g1_done, (uint32_t)(t & 1), 33);
        if constexpr (!PRO) {
          issue_x(0, g);
          issue_x(1, g + 1);
        }
      }
      mbar_wait(tfull, (uint32_t)(t & 1), 30);
      if (ew == 0) TRM(0, t, 2, TRM_CLK());
      tc_fence_after();
      // ---- pass 1: v = acc / 2 + b2 + x (the hidden operands are 2 GELU; PRO: acc already holds 2 x, no residual
      //      read); park v in TMEM, write it back to the residual stream, shifted statistics ----
      float s = 0.f, ss = 0.f, c0 = 0.f;
      long long p1_ld = 0, p1_sw = 0, p1_v = 0, p1_st = 0, p1_fence = 0, p1_tma = 0; (void)p1_ld; (void)p1_sw; (void)p1_v; (void)p1_st; (void)p1_fence; (void)p1_tma;
#pragma unroll 1
      for (int j = 0; j < CHUNKS; ++j, g += PRO ? 0 : 1) {
        const int col0 = c * NW + j * XW;
        const long long k0 = TRM_CLK(); (void)k0;
        uint32_t acc[XW];
        tmem_ld_cols(tlane + j * XW, acc);
        if constexpr (!PRO) mbar_wait(&my_xfull[g & 1], (uint32_t)(g >> 1) & 1u, 31);
        tmem_ld_wait();
        const long long k1 = TRM_CLK(); (void)k1;
        // shared-window addresses of this lane's row in the in-box / out-box (16-byte chunk i lives at swz_chunk(i))
        const uint32_t in_row = smem_u32(xbox) + (uint32_t)(g & 1) * Cfg::XBOX + lane * ROWB;
        const uint32_t out_row = smem_u32(obox) + lane * ROWB;
        const uint32_t bias_a = smem_u32(sBias) + col0 * 4;
        if (lane == 0) tma_store_wait_read();     // the previous chunk's store has finished reading the out-box
        __syncwarp();
        const long long k2 = TRM_CLK(); (void)k2;
        // first the updated row: it goes to the out-box at once, so that the stores have drained by the time the proxy
        // fence in front of the TMA store is reached (MEMBAR.ALL.CTA waits for every store in flight: ~300 cycles when it
        // came right behind the last store); the statistics are computed while they drain
#pragma unroll
        for (int i = 0; i < XW / 4; ++i) {
          const uint32_t off = swz_chunk<ROWB>(i, lane) << 4;
          const float4 b4 = lds_f4(bias_a + 16 * i);
          // packed fp32 pairs: the epilogue passes are issue bound (16 epilogue warps changed nothing), FADD2 / FFMA2
          // halve their arithmetic instructions
          float4 v;
          if constexpr (PRO) {
            f2_unpack(f2_fma(f2_from_bits(acc[4 * i + 0], acc[4 * i + 1]), f2_dup(0.5f), f2_pack(b4.x, b4.y)), v.x, v.y);
            f2_unpack(f2_fma(f2_from_bits(acc[4 * i + 2], acc[4 * i + 3]), f2_dup(0.5f), f2_pack(b4.z, b4.w)), v.z, v.w);
          } else {
            const float4 xv = lds_f4(in_row + off);
            f2_unpack(f2_fma(f2_from_bits(acc[4 * i + 0], acc[4 * i + 1]), f2_dup(0.5f), f2_add(f2_pack(b4.x, b4.y), f2_pack(xv.x, xv.y))), v.x, v.y);
            f2_unpack(f2_fma(f2_from_bits(acc[4 * i + 2], acc[4 * i + 3]), f2_dup(0.5f), f2_add(f2_pack(b4.z, b4.w), f2_pack(xv.z, xv.w))), v.z, v.w);
          }
          sts_f4(out_row + off, v);
          acc[4 * i + 0] = __float_as_uint(v.x); acc[4 * i + 1] = __float_as_uint(v.y);
          acc[4 * i + 2] = __float_as_uint(v.z); acc[4 * i + 3] = __float_as_uint(v.w);
        }
        if (j == 0) c0 = __uint_as_float(acc[0]);
        const long long k3 = TRM_CLK(); (void)k3;
        accum_stats(acc, c0, s, ss);
        const long long k4 = TRM_CLK(); (void)k4;
        tmem_st_cols(tlane + j * XW, acc);
        fence_proxy_async_smem();
        __syncwarp();                             // every lane has read the in-box and written the out-box
        const long long k5 = TRM_CLK(); (void)k5;
        if (lane == 0) {
          if (!PRO && j + 2 < CHUNKS) issue_x(j + 2, g + 2);   // refill the in-box right away (boxes never cross a tile here)
          tma_store_2d(&tmX, obox, col0, row0);
          tma_store_commit();
        }
        const long long k6 = TRM_CLK(); (void)k6;
        TR2_ACC(p1_ld, k0, k1); TR2_ACC(p1_sw, k1, k2); TR2_ACC(p1_v, k2, k3); TR2_ACC(p1_st, k3, k4); TR2_ACC(p1_fence, k4, k5);
        TR2_ACC(p1_tma, k5, k6);
      }
      tmem_st_wait();
      TR2(t, 0, p1_ld); TR2(t, 1, p1_sw); TR2(t, 2, p1_v); TR2(t, 3, p1_st); TR2(t, 4, p1_fence); TR2(t, 5, p1_tma);
      if (ew == 0) TRM(0, t, 3, TRM_CLK());
      // the residual boxes are done: once the last out-box store has been read, the h-tile producer may refill the region
      if (lane == 0) {
        tma_store_wait_read();
        fence_proxy_async_smem();
        mbar_arrive(a_free);
      }
      uint64_t nmean2, rstd2;
      row_stats(s, ss, c0, false, nmean2, rstd2);
      // ---- pass 2: normalise out of TMEM, fp16, 32-column chunks through the warp's staging box (64B-swizzled rows) ----
      const uint32_t hbox_a = smem_u32(hbox) + lane * 64, g_a = smem_u32(sG), bt_a = smem_u32(sBt);
      auto normalise_chunk = [&](const uint32_t (&v)[32], int j) {
        const int col0 = c * NW + j * 32;
        if (lane == 0) tma_store_wait_read();     // the previous chunk's store has finished reading the staging box
        __syncwarp();
#pragma unroll
        for (int i = 0; i < 4; ++i)
          sts_u4(hbox_a + (swz_chunk<64>(i, lane) << 4),
                 normalise8(v + 8 * i, g_a + col0 * 4 + 32 * i, bt_a + col0 * 4 + 32 * i, nmean2, rstd2));
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          tma_store_2d(&tmH, hbox, col0, row0);
          tma_store_commit();
        }
      };
      // (a two-register-buffer version with the TMEM read of chunk j + 1 in flight measured slower: 8.0 k vs 6.0 k
      //  cycles per tile; profiles/README.md)
#pragma unroll 1
      for (int j = 0; j < NW / 32; ++j) {
        uint32_t v[32];
        tmem_ld_32x32b_x32(tlane + j * 32, v);
        tmem_ld_wait();
        if (j == NW / 32 - 1) {
          // last read of this tile's accumulator: hand O back to the MMA warp
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_leader(tempty);
        }
        normalise_chunk(v, j);
      }
      if (ew == 0) TRM(0, t, 4, TRM_CLK());
      // the sPart exchange of the next tile must not overtake a slow partner still reading this tile's entry
      asm volatile("bar.sync %0, %1;" ::"r"(q + 1), "n"(32 * CG) : "memory");
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

bool mlp_resid_ln_supported(int M, int D, int hidden) {
  return D == LN_N && hidden >= HC && hidden % HC == 0 && hidden <= 8192 && M >= 1;
}

bool cproj_mlp_resid_ln_supported(int M, int D, int K, int hidden) {
  return mlp_resid_ln_supported(M, D, hidden) && K == D && MlpCfg<2>::smem_bytes(hidden, true) <= 232448;
}

// PRO: a_in = o and Wp / bproj / ln2_* the cross projection and norm2; otherwise a_in = h and those are unused
template <int CG, bool PRO>
static int mlp_ln_launch(const act_t* a_in, const act_t* Wp, const float* bproj, const float* ln2_w, const float* ln2_b,
                         const act_t* W1, const float* b1, const act_t* W2, const float* b2, float* x, const float* ln_w,
                         const float* ln_b, act_t* h_out, int M, int D, int hidden, float eps, cudaStream_t stream) {
  using Cfg = MlpCfg<CG>;
  const char* name = PRO ? "cproj_mlp_resid_ln" : "mlp_resid_ln";
  const int sms = gemm_num_sms();
  VITED_CHECK(sms >= 2, "%s: no device", name);
  const uint32_t smem = Cfg::smem_bytes(hidden, PRO);
  VITED_CHECK(smem <= 232448, "%s: hidden=%d needs %u bytes of shared memory", name, hidden, smem);
  static PerDeviceOnce once;
  if (once.first())
    VITED_CUDA_OK(cudaFuncSetAttribute(mlp_ln_pair_kernel<CG, PRO>, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448));
  CUtensorMap tA, tWp, tW1, tW2, tX, tH;
  if (make_tmap_act_2d(&tA, a_in, (uint64_t)D, (uint64_t)M, (uint64_t)D * 2, 64, BM, 128)) return 1;
  if (make_tmap_act_2d(&tW1, W1, (uint64_t)D, (uint64_t)hidden, (uint64_t)D * 2, 64, HC / 2, 128)) return 1;
  if (make_tmap_act_2d(&tW2, W2, (uint64_t)hidden, (uint64_t)D, (uint64_t)hidden * 2, 64, NH / 2, 128)) return 1;
  if (PRO) {
    if (make_tmap_act_2d(&tWp, Wp, (uint64_t)D, (uint64_t)D, (uint64_t)D * 2, 64, NH / 2, 128)) return 1;
  } else {
    tWp = tW1;
  }
  if (make_tmap_f32_2d(&tX, x, (uint64_t)D, (uint64_t)M, (uint64_t)D * 4, Cfg::XW, 32, Cfg::ROWB)) return 1;
  if (make_tmap_act_2d(&tH, h_out, (uint64_t)D, (uint64_t)M, (uint64_t)D * 2, 32, 32, 64)) return 1;
  const int tiles = (M + 2 * BM - 1) / (2 * BM);
  int pairs = sms / 2;
  if (pairs > tiles) pairs = tiles;
  VITED_CUDA_OK(launch_pdl(mlp_ln_pair_kernel<CG, PRO>, dim3(2 * pairs), dim3(Cfg::kThreads), smem, stream, tA, tWp, tW1,
                           tW2, tX, tH, bproj, ln2_w, ln2_b, b1, b2, ln_w, ln_b, M, hidden, eps));
  return 0;
}

int mlp_resid_ln(const act_t* h_in, const act_t* W1, const float* b1, const act_t* W2, const float* b2, float* x,
                 const float* ln_w, const float* ln_b, act_t* h_out, int M, int D, int hidden, float eps,
                 cudaStream_t stream) {
  VITED_CHECK(mlp_resid_ln_supported(M, D, hidden), "mlp_resid_ln: unsupported shape M=%d D=%d hidden=%d", M, D, hidden);
  VITED_CHECK(((reinterpret_cast<uintptr_t>(h_in) | reinterpret_cast<uintptr_t>(W1) | reinterpret_cast<uintptr_t>(W2) |
                reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(h_out)) & 15) == 0,
              "mlp_resid_ln: operands must be 16-byte aligned");
#ifdef VITED_EXPERIMENTAL   // measured neutral (profiles/README.md): not in the product library
  if (epilogue_warps() == 16)
    return mlp_ln_launch<4, false>(h_in, nullptr, nullptr, nullptr, nullptr, W1, b1, W2, b2, x, ln_w, ln_b, h_out, M, D,
                                   hidden, eps, stream);
#endif
  return mlp_ln_launch<2, false>(h_in, nullptr, nullptr, nullptr, nullptr, W1, b1, W2, b2, x, ln_w, ln_b, h_out, M, D,
                                 hidden, eps, stream);
}

int cproj_mlp_resid_ln(const act_t* o, const act_t* Wp, const float* bp, float* x, const float* ln2_w,
                       const float* ln2_b, const act_t* W1, const float* b1, const act_t* W2, const float* b2,
                       const float* ln_w, const float* ln_b, act_t* h_out, int M, int D, int hidden, float eps,
                       cudaStream_t stream) {
  VITED_CHECK(cproj_mlp_resid_ln_supported(M, D, D, hidden), "cproj_mlp_resid_ln: unsupported shape M=%d D=%d hidden=%d",
              M, D, hidden);
  VITED_CHECK(((reinterpret_cast<uintptr_t>(o) | reinterpret_cast<uintptr_t>(Wp) | reinterpret_cast<uintptr_t>(W1) |
                reinterpret_cast<uintptr_t>(W2) | reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(h_out)) &
               15) == 0,
              "cproj_mlp_resid_ln: operands must be 16-byte aligned");
  return mlp_ln_launch<2, true>(o, Wp, bp, ln2_w, ln2_b, W1, b1, W2, b2, x, ln_w, ln_b, h_out, M, D, hidden, eps, stream);
}

}  // namespace vited

#ifdef VITED_MLP_TRACE
extern "C" __attribute__((visibility("default"))) int vited_debug_mlp_trace(long long* out) {
  return (int)cudaMemcpyFromSymbol(out, vited::g_mlp_trace, sizeof(long long) * 2 * 32 * 8);
}
extern "C" __attribute__((visibility("default"))) int vited_debug_mlp_trace2(long long* out) {
  return (int)cudaMemcpyFromSymbol(out, vited::g_mlp_trace2, sizeof(long long) * 32 * 8);
}
#endif
