// Persistent, warp-specialised fp16 GEMM for sm_100a: TMA -> 128B-swizzled smem ring -> tcgen05.mma (accumulators
// in TMEM, double buffered) -> tcgen05.ld epilogue (bias / exact-erf GELU) -> swizzled smem staging -> TMA store.
//
// Computes what every Linear on the ViT-ED hot path computes (reference: models/vision_transformer.py:34,38 qkv/proj,
// :151-156 q/kv/proj, timm Mlp fc1/fc2, timm PatchEmbed conv-as-GEMM):  C = act(A * W^T + bias).
//   A [M,K] fp16 row-major (activations), W [N,K] fp16 row-major (PyTorch Linear layout) -> both operands K-major.
//
// Warp roles (128 + 32*4*BN/64 threads, 1 CTA / SM):
//   warp 0 lane 0 : TMA producer            warp 1 lane 0 : tcgen05.mma issuer
//   warp 2        : TMEM allocator          warps 4..     : epilogue; warp (q, sl) owns TMEM lane quarter q = warp%4
//                                             and the 64-column slab sl, stages its 32x64 fp16 sub-tile in a private
//                                             4 KB swizzled buffer and TMA-stores it itself (no CTA-wide barrier).
#include "kernels.h"
#include <cudaTypedefs.h>
#include <mutex>

namespace vited {

static PFN_cuTensorMapEncodeTiled_v12000 g_encode = nullptr;
static std::once_flag g_once;
static int g_init_status = 0;

int device_sm_count() {
  static int sms[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  int& n = sms[dev & 63];
  if (n == 0) cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
  return n;
}
#define g_num_sms device_sm_count()

static void init_driver_once() {
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
  if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || fn == nullptr) {
    set_error("cudaGetDriverEntryPoint(cuTensorMapEncodeTiled) failed: %s", cudaGetErrorString(e));
    g_init_status = 1;
    return;
  }
  g_encode = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(fn);
}

int gemm_num_sms() {
  std::call_once(g_once, init_driver_once);
  return device_sm_count();
}

// Every launch needs 3-6 tensor maps and a step makes ~7,500 launches over a handful of buffers and shapes that repeat
// chunk after chunk: encoded maps are kept in a small direct-mapped cache keyed by everything that goes into the
// encoding (a CUtensorMap is a pure function of these values, so a hit is always valid, also after the buffer was
// freed and another one allocated at the same address).
struct TmapKey {
  const void* ptr; uint64_t cols, rows, stride; uint32_t box_cols, box_rows; int32_t swizzle, dtype, promo;
  bool operator==(const TmapKey& o) const {
    return ptr == o.ptr && cols == o.cols && rows == o.rows && stride == o.stride && box_cols == o.box_cols &&
           box_rows == o.box_rows && swizzle == o.swizzle && dtype == o.dtype && promo == o.promo;
  }
};
struct TmapSlot { TmapKey key; CUtensorMap map; bool valid; };
constexpr int kTmapCacheSize = 1024;
static TmapSlot g_tmap_cache[kTmapCacheSize];
static std::mutex g_tmap_mutex;

static int encode_cached(CUtensorMap* tm, const TmapKey& k) {
  uint64_t h = reinterpret_cast<uint64_t>(k.ptr) * 0x9E3779B97F4A7C15ull;
  h ^= (k.cols * 0x100000001B3ull) ^ (k.rows * 0xC2B2AE3D27D4EB4Full) ^ (k.stride << 7) ^ ((uint64_t)k.box_cols << 40) ^
       ((uint64_t)k.box_rows << 48) ^ ((uint64_t)(k.swizzle * 4 + k.dtype * 2 + k.promo) << 56);
  h ^= h >> 29;
  std::lock_guard<std::mutex> lock(g_tmap_mutex);
  TmapSlot& sl = g_tmap_cache[h % kTmapCacheSize];
  if (sl.valid && sl.key == k) { *tm = sl.map; return 0; }
  cuuint64_t gdim[2] = {k.cols, k.rows};
  cuuint64_t gstride[1] = {k.stride};
  cuuint32_t box[2] = {k.box_cols, k.box_rows};
  cuuint32_t estr[2] = {1, 1};
  const CUtensorMapSwizzle sw = k.swizzle == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                                : k.swizzle == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_NONE;
  const CUtensorMapDataType dt = k.dtype == 2 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32
                                 : k.dtype == 1 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
  CUresult r = g_encode(tm, dt, 2, const_cast<void*>(k.ptr), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                        k.promo ? CU_TENSOR_MAP_L2_PROMOTION_L2_256B : CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (%d): ptr=%p cols=%llu rows=%llu stride=%llu box=%ux%u swizzle=%d dtype=%d",
              (int)r, k.ptr, (unsigned long long)k.cols, (unsigned long long)k.rows, (unsigned long long)k.stride,
              k.box_cols, k.box_rows, k.swizzle, k.dtype);
    return 1;
  }
  sl.key = k;
  sl.map = *tm;
  sl.valid = true;
  return 0;
}

// 2-D fp16 tensor map: inner dim = cols (contiguous), outer dim = rows, 128B swizzle, box = 64 cols x box_rows.
static int make_tmap(CUtensorMap* tm, const void* ptr, uint64_t cols, uint64_t rows, uint64_t row_stride_bytes,
                     uint32_t box_rows) {
  return encode_cached(tm, TmapKey{ptr, cols, rows, row_stride_bytes, 64, box_rows, 128, VITED_ACT_BF16, 1});
}
// generic 2-D fp16 tensor map for other kernels (attention): box = box_cols x box_rows, swizzle_bytes in {0, 64, 128}
int make_tmap_act_2d(CUtensorMap* tm, const void* ptr, uint64_t cols, uint64_t rows, uint64_t row_stride_bytes,
                      uint32_t box_cols, uint32_t box_rows, int swizzle_bytes) {
  std::call_once(g_once, init_driver_once);
  if (g_init_status) return 1;
  return encode_cached(tm, TmapKey{ptr, cols, rows, row_stride_bytes, box_cols, box_rows, swizzle_bytes, VITED_ACT_BF16, 0});
}

// 2-D fp32 tensor map (residual stream tiles of the fused GEMM + residual + LayerNorm kernels, gemm_ln.cu / mlp_ln.cu)
int make_tmap_f32_2d(CUtensorMap* tm, const void* ptr, uint64_t cols, uint64_t rows, uint64_t row_stride_bytes,
                     uint32_t box_cols, uint32_t box_rows, int swizzle_bytes) {
  std::call_once(g_once, init_driver_once);
  if (g_init_status) return 1;
  return encode_cached(tm, TmapKey{ptr, cols, rows, row_stride_bytes, box_cols, box_rows, swizzle_bytes, 2, 0});
}

constexpr int BM = 128;
constexpr int BK = 64;

template <int BN>
struct GemmCfg {
  static constexpr int kEpiWarps = 4 * (BN / 64);
  static constexpr int kThreads = 128 + 32 * kEpiWarps;
  static constexpr uint32_t A_BYTES = BM * BK * 2;
  static constexpr uint32_t B_BYTES = BN * BK * 2;
  static constexpr uint32_t STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr uint32_t C_BYTES = kEpiWarps * 4096;  // one 32-row x 128-byte swizzled box per epilogue warp
  static constexpr int kStagesMax = (232448 - 1024 - 256 - (int)C_BYTES) / (int)STAGE_BYTES;
  static constexpr int kStages = kStagesMax > 8 ? 8 : kStagesMax;
  static constexpr uint32_t TMEM_COLS = (2 * BN <= 256) ? 256 : 512;
  static constexpr uint32_t SMEM_BYTES = 1024 + kStages * STAGE_BYTES + C_BYTES + 256;
  static_assert(BN % 64 == 0 && BN <= 256, "BN must be a multiple of 64 up to 256");
  static_assert(kStages >= 3, "not enough shared memory for the pipeline");
};

// bias (+ GELU) on one thread's 64 accumulator columns, packed to fp16 and written into the warp's 32x128-byte staging
// box in the 128B-swizzle pattern the TMA store expects (16-byte chunk c of row r lives at chunk c ^ (r & 7)).
template <int ACT>
__device__ __forceinline__ void epilogue_tile(const uint32_t (&v0)[32], const uint32_t (&v1)[32],
                                              const float* __restrict__ bias, int n0, int N, uint8_t* rowp, int lane) {
  const uint32_t rowp_s = smem_u32(rowp);
#pragma unroll
  for (int ch = 0; ch < 2; ++ch) {
    const uint32_t* v = ch == 0 ? v0 : v1;
    const int nc = n0 + ch * 32;
    float f[32];
    if (nc + 32 <= N) {
#pragma unroll
      for (int i = 0; i < 8; ++i) {   // packed fp32 pairs: one FADD2 per two columns
        const float4 b4 = __ldg(reinterpret_cast<const float4*>(bias + nc) + i);
        f2_unpack(f2_add(f2_from_bits(v[4 * i + 0], v[4 * i + 1]), f2_pack(b4.x, b4.y)), f[4 * i + 0], f[4 * i + 1]);
        f2_unpack(f2_add(f2_from_bits(v[4 * i + 2], v[4 * i + 3]), f2_pack(b4.z, b4.w)), f[4 * i + 2], f[4 * i + 3]);
      }
    } else {
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        const float b = (nc + i < N) ? __ldg(bias + nc + i) : 0.f;
        f[i] = __uint_as_float(v[i]) + b;
      }
    }
    if (ACT == ACT_GELU) {
#pragma unroll
      for (int i = 0; i < 32; ++i) f[i] = gelu_fast(f[i]);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      uint4 pk;
      pk.x = pack_act(f[8 * i + 0], f[8 * i + 1]);
      pk.y = pack_act(f[8 * i + 2], f[8 * i + 3]);
      pk.z = pack_act(f[8 * i + 4], f[8 * i + 5]);
      pk.w = pack_act(f[8 * i + 6], f[8 * i + 7]);
      sts_u4(rowp_s + (((ch * 4 + i) ^ (lane & 7)) << 4), pk);   // explicit st.shared on a 32-bit address
    }
  }
}

template <int BN, int ACT>
__global__ void __launch_bounds__(GemmCfg<BN>::kThreads, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const __grid_constant__ CUtensorMap tmC, const float* __restrict__ bias, int M, int N, int K) {
  using Cfg = GemmCfg<BN>;
  constexpr int kStages = Cfg::kStages;
  constexpr int kEpiWarps = Cfg::kEpiWarps;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sC = smem + kStages * Cfg::STAGE_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sC + Cfg::C_BYTES);
  uint64_t* full = bars;
  uint64_t* empty = bars + kStages;
  uint64_t* tfull = bars + 2 * kStages;
  uint64_t* tempty = bars + 2 * kStages + 2;
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(bars + 2 * kStages + 4);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  const int m_blks = (M + BM - 1) / BM;
  const int n_blks = (N + BN - 1) / BN;
  const int num_kb = (K + BK - 1) / BK;
  // Tile schedule: tile = blockIdx.x + i*gridDim.x, n fastest.
  auto coords = [&](int it, int& m_blk, int& n_blk) -> bool {
    const int tile = (int)blockIdx.x + it * (int)gridDim.x;
    m_blk = tile / n_blks;
    n_blk = tile % n_blks;
    return tile < m_blks * n_blks;
  };

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    tma_prefetch_desc(&tmC);
  } else if (warp == 1 && lane == 0) {
    for (int s = 0; s < kStages; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tfull[s], 1);
      mbar_init(&tempty[s], kEpiWarps);
    }
    fence_mbar_init();
  } else if (warp == 2) {
    tmem_alloc(tmem_holder, Cfg::TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      uint32_t stage = 0, phase = 0;
      int m_blk, n_blk;
      for (int it = 0; coords(it, m_blk, n_blk); ++it) {
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&empty[stage], phase ^ 1, 10);
          uint8_t* a_dst = smem + stage * Cfg::STAGE_BYTES;
          mbar_arrive_expect_tx(&full[stage], Cfg::STAGE_BYTES);
          tma_load_2d(&tmA, &full[stage], a_dst, kb * BK, m_blk * BM);
          tma_load_2d(&tmB, &full[stage], a_dst + Cfg::A_BYTES, kb * BK, n_blk * BN);
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    // warp-uniform loop, tcgen05 instructions predicated on one elected lane (see elect_one_sync)
    {
      constexpr uint32_t idesc = umma_idesc_f16(BM, BN);
      uint32_t stage = 0, phase = 0, as = 0, aphase = 0;
      int m_blk, n_blk;
      for (int it = 0; coords(it, m_blk, n_blk); ++it) {
        mbar_wait(&tempty[as], aphase ^ 1, 20);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * BN;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&full[stage], phase, 21);
          tc_fence_after();
          const uint32_t lo_a = umma_desc_sw128_lo(smem_u32(smem)) + stage * (Cfg::STAGE_BYTES >> 4);
          const uint32_t lo_b = lo_a + (Cfg::A_BYTES >> 4);
          if (elect_one_sync()) {
#pragma unroll
            for (int k = 0; k < BK / 16; ++k) {
              // advance 16 fp16 = 32 B along K inside the 128B swizzle atom: +2 in the (addr >> 4) field
              umma_f16(d_tmem, umma_desc_pack(lo_a + 2 * k, kUmmaDescSw128Hi), umma_desc_pack(lo_b + 2 * k, kUmmaDescSw128Hi),
                        idesc, (kb | k) != 0 ? 1u : 0u);
            }
            umma_commit(&empty[stage]);  // frees the smem stage once these MMAs have read it
          }
          __syncwarp();
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
        if (elect_one_sync()) umma_commit(&tfull[as]);  // accumulator complete -> epilogue
        __syncwarp();
        if (++as == 2) { as = 0; aphase ^= 1; }
      }
    }
  } else if (warp >= 4) {
    // ===================== epilogue =====================
    const int ew = warp - 4;
    const int q = warp & 3;   // TMEM lane quarter this warp may read
    const int sl = ew >> 2;   // 64-column slab of the tile
    uint8_t* my_stage = sC + ew * 4096;          // 32 rows x 128 B, 128B-swizzled (what the TMA store box expects)
    uint8_t* rowp = my_stage + lane * 128;
    uint32_t as = 0, aphase = 0;
    bool store_pending = false;
    int m_blk, n_blk;
    for (int it = 0; coords(it, m_blk, n_blk); ++it) {
      const int n0 = n_blk * BN + sl * 64;
      mbar_wait(&tfull[as], aphase, 30);
      tc_fence_after();
      uint32_t v0[32], v1[32];
      const uint32_t taddr = tmem_base + as * BN + sl * 64 + (static_cast<uint32_t>(q * 32) << 16);
      tmem_ld_32x32b_x32(taddr, v0);
      tmem_ld_32x32b_x32(taddr + 32, v1);
      tmem_ld_wait();
      // accumulator values are in registers: hand the TMEM stage back to the MMA warp right away
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty[as]);
      // the previous tile's TMA store must have finished reading this warp's staging buffer
      if (store_pending) {
        if (lane == 0) tma_store_wait_read();
        __syncwarp();
      }
      epilogue_tile<ACT>(v0, v1, bias, n0, N, rowp, lane);
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0 && n0 < N) {
        tma_store_2d(&tmC, my_stage, n0, m_blk * BM + q * 32);
        tma_store_commit();
      }
      store_pending = true;
      if (++as == 2) { as = 0; aphase ^= 1; }
    }
    if (lane == 0) tma_store_wait_all();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
  }
}

// =====================================================================================================================
// CTA-pair variant (cta_group::2): the two CTAs of a cluster compute one 256 x BN tile. Each CTA streams its own 128
// activation rows and HALF of the weight tile; tcgen05.mma.cta_group::2 (issued by the leader CTA) reads both halves,
// so the weight bytes every SM has to pull through its TMA ring and shared memory are halved. With K = 384 the ring
// (bytes in flight per SM) is what limits the single-CTA kernel (profiles/: tensor pipe ~60 %, nothing saturated).
// =====================================================================================================================
template <int BN>
struct PairCfg {
  static constexpr int kEpiWarps = 4 * (BN / 64);
  static constexpr int kThreads = 128 + 32 * kEpiWarps;
  static constexpr uint32_t A_BYTES = BM * BK * 2;
  static constexpr uint32_t BH_BYTES = (BN / 2) * BK * 2;     // this CTA's half of the weight tile
  static constexpr uint32_t STAGE_BYTES = A_BYTES + BH_BYTES;
  static constexpr uint32_t C_BYTES = kEpiWarps * 4096;
  static constexpr int kStagesMax = (232448 - 1024 - 256 - (int)C_BYTES) / (int)STAGE_BYTES;
  static constexpr int kStages = kStagesMax > 8 ? 8 : kStagesMax;
  static constexpr uint32_t TMEM_COLS = (2 * BN <= 256) ? 256 : 512;
  static constexpr uint32_t SMEM_BYTES = 1024 + kStages * STAGE_BYTES + C_BYTES + 256;
  static_assert(BN % 64 == 0 && BN <= 256 && (BN / 2) % 8 == 0, "bad BN");
  static_assert(kStages >= 3, "not enough shared memory for the pipeline");
};

template <int BN, int ACT>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(PairCfg<BN>::kThreads, 1)
gemm_tc_pair_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                    const __grid_constant__ CUtensorMap tmC, const float* __restrict__ bias, int M, int N, int K) {
  using Cfg = PairCfg<BN>;
  constexpr int kStages = Cfg::kStages;
  constexpr int kEpiWarps = Cfg::kEpiWarps;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sC = smem + kStages * Cfg::STAGE_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sC + Cfg::C_BYTES);
  uint64_t* full = bars;                     // used in the leader CTA only (both CTAs' TMA bytes land on it)
  uint64_t* empty = bars + kStages;          // per CTA, released by the leader's multicast commit
  uint64_t* tfull = bars + 2 * kStages;      // per CTA, multicast commit
  uint64_t* tempty = bars + 2 * kStages + 2; // leader CTA only: epilogue warps of BOTH CTAs arrive
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(bars + 2 * kStages + 4);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int pair = (int)(blockIdx.x >> 1);
  const int num_pairs = (int)(gridDim.x >> 1);

  const int m2_blks = (M + 2 * BM - 1) / (2 * BM);
  const int n_blks = (N + BN - 1) / BN;
  const int num_tiles = m2_blks * n_blks;
  const int num_kb = (K + BK - 1) / BK;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    tma_prefetch_desc(&tmC);
  } else if (warp == 1 && lane == 0) {
    for (int s = 0; s < kStages; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tfull[s], 1);
      mbar_init(&tempty[s], 2 * kEpiWarps);
    }
    fence_mbar_init();
  } else if (warp == 2) {
    tmem_alloc_2cta(tmem_holder, Cfg::TMEM_COLS);
    tmem_relinquish_2cta();
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();   // the peer's barriers exist before anything is signalled across the pair
  tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;

  if (warp == 0) {
    // ===================== TMA producer (both CTAs) =====================
    if (lane == 0) {
      uint32_t stage = 0, phase = 0;
      for (int tile = pair; tile < num_tiles; tile += num_pairs) {
        const int m2 = tile / n_blks, n_blk = tile % n_blks;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&empty[stage], phase ^ 1, 10);
          uint8_t* a_dst = smem + stage * Cfg::STAGE_BYTES;
          if (rank == 0) mbar_arrive_expect_tx(&full[stage], 2 * Cfg::STAGE_BYTES);
          tma_load_2d_2cta(&tmA, &full[stage], a_dst, kb * BK, m2 * 2 * BM + (int)rank * BM);
          tma_load_2d_2cta(&tmB, &full[stage], a_dst + Cfg::A_BYTES, kb * BK, n_blk * BN + (int)rank * (BN / 2));
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA only) =====================
    // The whole warp runs the loop (warp-uniform control flow and descriptors); only the tcgen05 instructions are
    // predicated on one elected lane.
    if (rank == 0) {
      constexpr uint32_t idesc = umma_idesc_f16(2 * BM, BN);
      constexpr uint32_t kStage16 = Cfg::STAGE_BYTES >> 4, kA16 = Cfg::A_BYTES >> 4;
      const uint32_t lo0 = umma_desc_sw128_lo(smem_u32(smem));   // A tile of stage 0; the B half tile follows it
      uint32_t stage = 0, phase = 0, as = 0, aphase = 0;
      for (int tile = pair; tile < num_tiles; tile += num_pairs) {
        mbar_wait(&tempty[as], aphase ^ 1, 20);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * BN;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&full[stage], phase, 21);
          tc_fence_after();
          const uint32_t lo_a = lo0 + stage * kStage16;
          if (elect_one_sync()) {
#pragma unroll
            for (int k = 0; k < BK / 16; ++k)   // 16 fp16 = 32 B along K inside the swizzle atom: +2 in the address field
              umma_f16_2cta(d_tmem, umma_desc_pack(lo_a + 2 * k, kUmmaDescSw128Hi),
                             umma_desc_pack(lo_a + kA16 + 2 * k, kUmmaDescSw128Hi), idesc, (kb | k) != 0 ? 1u : 0u);
            umma_commit_2cta(&empty[stage]);   // frees this stage in BOTH CTAs
          }
          __syncwarp();
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
        if (elect_one_sync()) umma_commit_2cta(&tfull[as]);        // accumulators complete in BOTH CTAs
        __syncwarp();
        if (++as == 2) { as = 0; aphase ^= 1; }
      }
    }
  } else if (warp >= 4) {
    // ===================== epilogue (both CTAs, own 128 rows) =====================
    const int ew = warp - 4;
    const int q = warp & 3;
    const int sl = ew >> 2;
    uint8_t* my_stage = sC + ew * 4096;
    uint8_t* rowp = my_stage + lane * 128;
    uint32_t as = 0, aphase = 0;
    bool store_pending = false;
    for (int tile = pair; tile < num_tiles; tile += num_pairs) {
      const int m2 = tile / n_blks, n_blk = tile % n_blks;
      const int n0 = n_blk * BN + sl * 64;
      mbar_wait(&tfull[as], aphase, 30);
      tc_fence_after();
      uint32_t v0[32], v1[32];
      const uint32_t taddr = tmem_base + as * BN + sl * 64 + (static_cast<uint32_t>(q * 32) << 16);
      tmem_ld_32x32b_x32(taddr, v0);
      tmem_ld_32x32b_x32(taddr + 32, v1);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_leader(&tempty[as]);
      if (store_pending) {
        if (lane == 0) tma_store_wait_read();
        __syncwarp();
      }
      epilogue_tile<ACT>(v0, v1, bias, n0, N, rowp, lane);
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0 && n0 < N) {
        tma_store_2d(&tmC, my_stage, n0, m2 * 2 * BM + (int)rank * BM + q * 32);
        tma_store_commit();
      }
      store_pending = true;
      if (++as == 2) { as = 0; aphase ^= 1; }
    }
    if (lane == 0) tma_store_wait_all();
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();   // neither CTA may leave (or free TMEM) while the other can still touch its barriers / smem
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc_2cta(tmem_base, Cfg::TMEM_COLS);
  }
}

template <int BN, int ACT>
static int launch_pair(const CUtensorMap& tA, const CUtensorMap& tB, const CUtensorMap& tC, const float* bias, int M,
                       int N, int K, cudaStream_t stream) {
  using Cfg = PairCfg<BN>;
  static PerDeviceOnce once;
  if (once.first())
    VITED_CUDA_OK(cudaFuncSetAttribute(gemm_tc_pair_kernel<BN, ACT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)Cfg::SMEM_BYTES));
  const int tiles = ((M + 2 * BM - 1) / (2 * BM)) * ((N + BN - 1) / BN);
  int pairs = g_num_sms / 2;
  if (pairs > tiles) pairs = tiles;
  gemm_tc_pair_kernel<BN, ACT><<<2 * pairs, Cfg::kThreads, Cfg::SMEM_BYTES, stream>>>(tA, tB, tC, bias, M, N, K);
  VITED_CUDA_OK(cudaGetLastError());
  return 0;
}

template <int BN, int ACT>
static int launch_tc(const CUtensorMap& tA, const CUtensorMap& tB, const CUtensorMap& tC, const float* bias, int M,
                     int N, int K, cudaStream_t stream) {
  using Cfg = GemmCfg<BN>;
  static PerDeviceOnce once;
  if (once.first())
    VITED_CUDA_OK(cudaFuncSetAttribute(gemm_tc_kernel<BN, ACT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)Cfg::SMEM_BYTES));
  const int tiles = ((M + BM - 1) / BM) * ((N + BN - 1) / BN);
  const int grid = tiles < g_num_sms ? tiles : g_num_sms;
  gemm_tc_kernel<BN, ACT><<<grid, Cfg::kThreads, Cfg::SMEM_BYTES, stream>>>(tA, tB, tC, bias, M, N, K);
  VITED_CUDA_OK(cudaGetLastError());
  return 0;
}

template <int BN>
static int launch_act(const CUtensorMap& tA, const CUtensorMap& tB, const CUtensorMap& tC, const float* bias, int M,
                      int N, int K, int act, cudaStream_t stream) {
  return act == ACT_GELU ? launch_tc<BN, ACT_GELU>(tA, tB, tC, bias, M, N, K, stream)
                         : launch_tc<BN, ACT_NONE>(tA, tB, tC, bias, M, N, K, stream);
}

int gemm_simt(const act_t* A, const act_t* W, const float* bias, act_t* C, int M, int N, int K, int act,
              cudaStream_t stream);

int gemm_act(const act_t* A, const act_t* W, const float* bias, act_t* C, int M, int N, int K, int act, int impl,
              cudaStream_t stream) {
  VITED_CHECK(M > 0 && N > 0 && K > 0, "gemm_act: empty problem M=%d N=%d K=%d", M, N, K);
  if (impl == IMPL_REF) return gemm_simt(A, W, bias, C, M, N, K, act, stream);
  std::call_once(g_once, init_driver_once);
  if (g_init_status) return 1;
  VITED_CHECK(K % 8 == 0 && N % 8 == 0, "gemm_act: K and N must be multiples of 8 (TMA 16-byte strides), got K=%d N=%d",
              K, N);
  VITED_CHECK((reinterpret_cast<uintptr_t>(A) & 15) == 0 && (reinterpret_cast<uintptr_t>(W) & 15) == 0 &&
                  (reinterpret_cast<uintptr_t>(C) & 15) == 0,
              "gemm_act: operands must be 16-byte aligned");
  // Tile width: the widest of 256 / 192 / 128 that divides N. Large M (at least two 128-row blocks per SM) goes to the
  // CTA-pair kernel when N takes a 256- or 192-wide tile.
  const int m_blks = (M + BM - 1) / BM;
  const int bn = N % 256 == 0 ? 256 : N % 192 == 0 ? 192 : 128;
  CUtensorMap tA, tB, tC;
  if (make_tmap(&tA, A, (uint64_t)K, (uint64_t)M, (uint64_t)K * 2, BM)) return 1;
  if (bn != 128 && m_blks >= 2 * g_num_sms) {
    if (make_tmap(&tB, W, (uint64_t)K, (uint64_t)N, (uint64_t)K * 2, (uint32_t)bn / 2)) return 1;
    if (make_tmap(&tC, C, (uint64_t)N, (uint64_t)M, (uint64_t)N * 2, 32)) return 1;
    if (bn == 256)
      return act == ACT_GELU ? launch_pair<256, ACT_GELU>(tA, tB, tC, bias, M, N, K, stream)
                             : launch_pair<256, ACT_NONE>(tA, tB, tC, bias, M, N, K, stream);
    return act == ACT_GELU ? launch_pair<192, ACT_GELU>(tA, tB, tC, bias, M, N, K, stream)
                           : launch_pair<192, ACT_NONE>(tA, tB, tC, bias, M, N, K, stream);
  }
  if (make_tmap(&tB, W, (uint64_t)K, (uint64_t)N, (uint64_t)K * 2, (uint32_t)bn)) return 1;
  if (make_tmap(&tC, C, (uint64_t)N, (uint64_t)M, (uint64_t)N * 2, 32)) return 1;
  if (bn == 128) return launch_act<128>(tA, tB, tC, bias, M, N, K, act, stream);
  if (bn == 256) return launch_act<256>(tA, tB, tC, bias, M, N, K, act, stream);
  return launch_act<192>(tA, tB, tC, bias, M, N, K, act, stream);
}

}  // namespace vited
