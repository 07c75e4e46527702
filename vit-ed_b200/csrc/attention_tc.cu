// tcgen05 attention kernels for the two hot decoder shapes (reference: models/vision_transformer.py:56-80
// Attention.forward, :174-200 CrossAttention.forward; SDPA scale head_dim^-0.5, no mask, eval mode).
//
// attn_p64_kernel -- puzzle model: 64 patch tokens (+ class token) per sequence, head_dim 32.
//   One work unit = one (sequence, head): S = Q K^T is ONE 128 x {64|80} tcgen05.mma pair (rows 0..63 = patch queries,
//   row 64 = the class-token query, rows 65..127 unused), softmax runs with one thread per query row straight out of
//   TMEM, the probabilities go back to TMEM as packed fp16 (aliasing S) and feed the second MMA as its A operand,
//   O = P V with V consumed in place as an MN-major operand (no transpose, no ldmatrix, no shuffles).
//   Warp roles (16 warps, 1 CTA / SM): warp 3 = TMA producer (12-deep ring of Q/K/V tiles, hardware 64B swizzle),
//   warp 7 = MMA issuer (lean, warp-uniform, serves the groups' units in round-robin order: PV of a unit, then QK^T
//   of the same group's next unit right behind it), warp 11 = TMEM allocator, warps {4g, 4g+1, 4g+2} = softmax group g
//   of TMEM stage g (rows 0-31, 32-63, 64).
// Operand conventions (SW64 K-major, MN-major V, A from TMEM) were pinned on B200 by tools/umma_probe.cu.
#include "kernels.h"

namespace vited {

namespace {

constexpr float kLog2e = 1.4426950408889634f;

__device__ __forceinline__ float ex2_ftz(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

struct P64 {
  static constexpr int HD = 32;
  static constexpr int RB = 64;               // bytes per tile row
  static constexpr int TROWS = 80;            // 64 patch rows + class-token row (64) + 15 zero rows
  static constexpr int TB = TROWS * RB;       // 5120
  static constexpr int STAGE = 3 * TB;        // Q, K, V
  static constexpr int NS = 12;               // shared-memory ring depth (units in flight)
  static constexpr int NT = 4;                // TMEM stages = softmax groups
  static constexpr int TCOLS = 128;           // TMEM columns per stage: S/P at +0 (80), O at +96 (32)
  static constexpr int OCOL = 96;
  static constexpr int THREADS = 32 * 4 * NT;
  static constexpr int BAR_BYTES = (2 * NS + 4 * NT) * 8 + 16;   // full, empty, s_full, o_full, p_ready + TMEM holder
  static constexpr int BYTES = 1024 + NS * STAGE + BAR_BYTES;
};

#ifdef VITED_ATTN_TRACE   // clock64 trace of block 0 (tools/trace_attn_p64.py); compiled out of the product library
__device__ unsigned long long g_p64_trace[4 * 64 * 8];   // [group][unit k][event], first warp lane 0
#define TRP(ev) do { if (blockIdx.x == 0 && quarter == 0 && lane == 0 && tk < 64) g_p64_trace[(group * 64 + tk) * 8 + (ev)] = clock64(); } while (0)
#else
#define TRP(ev) do { } while (0)
#endif

struct P64Maps {
  CUtensorMap q_tile, q_row, k_tile, k_row, v_tile, v_row;   // boxes {32, 64} and {32, 1}, 64B swizzle
};

__global__ void __launch_bounds__(P64::THREADS, 1)
attn_p64_kernel(AttnArgs a, const __grid_constant__ P64Maps maps, int n_units) {
  using C = P64;
  extern __shared__ uint8_t attn_tc_smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(attn_tc_smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + C::NS * C::STAGE);
  uint64_t* full = bars;                       // TMA bytes landed (count 1 + tx)
  uint64_t* empty = bars + C::NS;              // PV of the unit has read the stage (tcgen05.commit)
  uint64_t* s_full = bars + 2 * C::NS;         // S ready in TMEM (commit)
  uint64_t* o_full = s_full + C::NT;           // O ready in TMEM (commit)
  uint64_t* p_ready = o_full + C::NT;          // P written to TMEM (the group's 3 softmax warps)
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(p_ready + C::NT);

  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);   // provably warp-uniform (keeps MMA operands in uniform registers)
  const int quarter = warp & 3, group = warp >> 2;
  const int H = a.n_heads;
  const int n_my = (n_units - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  const int NK = a.k_has_cls ? 80 : 64;        // key columns of S (64 patch keys [+ class-token key + 15 zero rows])

  // rows 64..79 of every tile: the class-token row is TMA-written when present, everything else must be exact zeros
  for (int i = tid; i < C::NS * 3 * (16 * C::RB / 16); i += C::THREADS) {
    const int tile = i / (16 * C::RB / 16), r = i % (16 * C::RB / 16);
    *reinterpret_cast<uint4*>(smem + tile * C::TB + 64 * C::RB + r * 16) = make_uint4(0, 0, 0, 0);
  }
  if (tid == 0) {
    for (int s = 0; s < C::NS; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    for (int t = 0; t < C::NT; ++t) {
      mbar_init(&s_full[t], 1); mbar_init(&o_full[t], 1); mbar_init(&p_ready[t], 3);
    }
    fence_mbar_init();
    tma_prefetch_desc(&maps.q_tile);
    tma_prefetch_desc(&maps.k_tile);
    tma_prefetch_desc(&maps.v_tile);
  }
  if (warp == 11) {
    tmem_alloc(tmem_holder, 512);
    tmem_relinquish();
  }
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;

  if (quarter == 3) {
    if (group == 0) {
      // ===================== TMA producer =====================
      // Lane 0 issues. With a key/value index (cross-attention: kv_index[b]) the whole warp fetches the indices of the
      // next 32 units at once. A dependent __ldg per unit in the issuing thread's chain (~600 cycles) was the whole per-unit
      // budget of the cross-attention launch (~880 cycles per unit and SM).
      int s = 0;
      uint32_t ph = 0;
      auto issue_unit = [&](int i, int kvb) {     // lane 0: the TMA loads of local unit i
        const int u = (int)blockIdx.x + i * (int)gridDim.x;
        const int b = u / H, h = u - b * H;
        if (kvb < 0) kvb = b;
        const int col = h * C::HD;
        mbar_wait(&empty[s], ph ^ 1, 50);
        uint8_t* st = smem + s * C::STAGE;
        const uint32_t bytes = 3 * 64 * C::RB + (a.q_has_cls ? C::RB : 0) + (a.k_has_cls ? 2 * C::RB : 0);
        mbar_arrive_expect_tx(&full[s], bytes);
        tma_load_2d(&maps.q_tile, &full[s], st, col, b * 64);
        if (a.q_has_cls) tma_load_2d(&maps.q_row, &full[s], st + 64 * C::RB, col, a.n_seq * 64 + b);
        tma_load_2d(&maps.k_tile, &full[s], st + C::TB, col, kvb * 64);
        tma_load_2d(&maps.v_tile, &full[s], st + 2 * C::TB, col, kvb * 64);
        if (a.k_has_cls) {
          tma_load_2d(&maps.k_row, &full[s], st + C::TB + 64 * C::RB, col, a.n_kv_seq * 64 + kvb);
          tma_load_2d(&maps.v_row, &full[s], st + 2 * C::TB + 64 * C::RB, col, a.n_kv_seq * 64 + kvb);
        }
        if (++s == C::NS) { s = 0; ph ^= 1; }
      };
      if (a.kv_index == nullptr) {
        if (lane == 0)
          for (int i = 0; i < n_my; ++i) issue_unit(i, -1);
      } else {
        for (int i0 = 0; i0 < n_my; i0 += 32) {
          int my_kvb = 0;
          if (i0 + lane < n_my) my_kvb = __ldg(a.kv_index + ((int)blockIdx.x + (i0 + lane) * (int)gridDim.x) / H);
          const int jn = n_my - i0 < 32 ? n_my - i0 : 32;
          for (int j = 0; j < jn; ++j) {
            const int kvb = __shfl_sync(0xffffffffu, my_kvb, j);
            if (lane == 0) issue_unit(i0 + j, kvb);
          }
        }
      }
    } else if (group == 1) {
      // ===================== MMA issuer for all four groups (warp-uniform code, one elected lane) =====================
      // Units go to the groups round robin, so the issuer serves them in unit order: PV(i) as soon as the group's
      // probabilities are in TMEM, QK^T of the same group's next unit (i + NT) right behind it (the tensor pipe runs in
      // issue order, so those scores may overwrite P(i)). When the groups' first warps issued their own MMAs that cost
      // them ~850 cycles per unit on the group's critical path (tools/trace_attn_p64.py).
      const uint32_t idesc_qk = umma_idesc_f16(128, NK);
      const uint32_t idesc_pv = umma_idesc_f16(128, C::HD) | kIdescBMajorMN;
      const uint32_t smem0 = smem_u32(smem);
      auto issue_qk = [&](int i) {      // S(stage i % NT) = Q K^T of local unit i
        const int s = i % C::NS, t = i % C::NT;
        mbar_wait(&full[s], (uint32_t)(i / C::NS) & 1u, 51);
        tc_fence_after();
        const uint32_t q_addr = smem0 + s * C::STAGE;
        const uint64_t dq = umma_desc_sw(q_addr, 64);
        const uint64_t dk = umma_desc_sw(q_addr + C::TB, 64);
        const uint32_t t_col = tmem_base + t * C::TCOLS;
        if (elect_one_sync()) {
#pragma unroll
          for (int k = 0; k < C::HD / 16; ++k) umma_f16(t_col, dq + 2 * k, dk + 2 * k, idesc_qk, k);
          umma_commit(&s_full[t]);
        }
        __syncwarp();
      };
      for (int i = 0; i < C::NT && i < n_my; ++i) issue_qk(i);
      for (int i = 0; i < n_my; ++i) {
        const int s = i % C::NS, t = i % C::NT;
        const uint32_t t_col = tmem_base + t * C::TCOLS;
        mbar_wait(&p_ready[t], (uint32_t)(i / C::NT) & 1u, 53);
        tc_fence_after();
        const uint64_t dv = umma_desc_sw(smem0 + s * C::STAGE + 2 * C::TB, 64);
        if (elect_one_sync()) {
          if (NK == 80) {
#pragma unroll
            for (int k = 0; k < 5; ++k)   // 16 keys per step = two 8-key groups of 512 B = +64 in the (addr >> 4) field
              umma_f16_ts(t_col + C::OCOL, t_col + 8 * k, dv + 64 * k, idesc_pv, k);
          } else {
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma_f16_ts(t_col + C::OCOL, t_col + 8 * k, dv + 64 * k, idesc_pv, k);
          }
          umma_commit(&empty[s]);
          umma_commit(&o_full[t]);
        }
        __syncwarp();
        if (i + C::NT < n_my) issue_qk(i + C::NT);
      }
    }
  } else {
    // ===================== softmax group `group`, TMEM lane quarter `quarter` =====================
    // The group owns TMEM stage `group`: scores -> probabilities (packed fp16 over S) -> signal the issuer -> read O.
    const float sl2 = a.scale * kLog2e;
    const int row = quarter * 32 + lane;                  // query row of the unit's tile
    // quarter 2 only carries the class-token query (row 64)
    const bool warp_active = quarter < 2 || a.q_has_cls != 0;
    const uint32_t t_col = tmem_base + group * C::TCOLS;
    const uint32_t t_stage = t_col + (static_cast<uint32_t>(quarter * 32) << 16);
    uint32_t ph = 0;
    int tk = 0; (void)tk;
    for (int i = group; i < n_my; i += C::NT, ++tk) {
      const int u = (int)blockIdx.x + i * (int)gridDim.x;
      const int b = u / H, h = u - b * H;
      TRP(0);
      mbar_wait(&s_full[group], ph, 54);
      TRP(1);
      tc_fence_after();
      float l = 1.f;
      if (warp_active) {
        uint32_t v0[32], v1[32];
        uint32_t vc[8];
        tmem_ld_32x32b_x32(t_stage, v0);
        tmem_ld_32x32b_x32(t_stage + 32, v1);
        if (a.k_has_cls) tmem_ld_32x32b_x8(t_stage + 64, vc);
        tmem_ld_wait();
        float mx[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) mx[j] = fmaxf(__uint_as_float(v0[j]), __uint_as_float(v1[j]));
#pragma unroll
        for (int j = 4; j < 32; ++j) mx[j & 3] = fmaxf(mx[j & 3], fmaxf(__uint_as_float(v0[j]), __uint_as_float(v1[j])));
        float mxa = fmaxf(fmaxf(mx[0], mx[1]), fmaxf(mx[2], mx[3]));
        if (a.k_has_cls) mxa = fmaxf(mxa, __uint_as_float(vc[0]));
        const float mneg = -mxa * sl2;
        float sum[4] = {0.f, 0.f, 0.f, 0.f};
        uint32_t pk[32];
        {
          uint64_t sum2[2] = {0ull, 0ull};
          softmax_exp_pairs<16>(v0, sl2, mneg, pk, sum2);
          softmax_exp_pairs<16>(v1, sl2, mneg, pk + 16, sum2);
          f2_unpack(sum2[0], sum[0], sum[1]);
          f2_unpack(sum2[1], sum[2], sum[3]);
        }
        tmem_st_32x32b_x32(t_stage, pk);
        if (a.k_has_cls) {
          const float pc = ex2_ftz(fmaf(__uint_as_float(vc[0]), sl2, mneg));
          sum[0] += pc;
          uint32_t pc8[8] = {pack_act(pc, 0.f), 0u, 0u, 0u, 0u, 0u, 0u, 0u};
          tmem_st_32x32b_x8(t_stage + 32, pc8);
        }
        l = (sum[0] + sum[1]) + (sum[2] + sum[3]);
        tmem_st_wait();
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&p_ready[group]);   // 3 warps: all of P is in TMEM -> the issuer may run PV
      TRP(2);
      mbar_wait(&o_full[group], ph, 55);
      TRP(3);
      tc_fence_after();
      if (warp_active) {
        uint32_t ov[32];
        tmem_ld_32x32b_x32(t_stage + C::OCOL, ov);
        tmem_ld_wait();
        const float inv = 1.f / l;
        size_t orow;
        bool valid = true;
        if (row < 64) orow = (size_t)b * 64 + row;
        else if (row == 64 && a.q_has_cls) orow = (size_t)a.n_seq * 64 + b;
        else { valid = false; orow = 0; }
        if (valid) {
          uint4* dst = reinterpret_cast<uint4*>(a.o + orow * a.o_ld + h * C::HD);
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            uint4 w;
            w.x = pack_act(__uint_as_float(ov[8 * c + 0]) * inv, __uint_as_float(ov[8 * c + 1]) * inv);
            w.y = pack_act(__uint_as_float(ov[8 * c + 2]) * inv, __uint_as_float(ov[8 * c + 3]) * inv);
            w.z = pack_act(__uint_as_float(ov[8 * c + 4]) * inv, __uint_as_float(ov[8 * c + 5]) * inv);
            w.w = pack_act(__uint_as_float(ov[8 * c + 6]) * inv, __uint_as_float(ov[8 * c + 7]) * inv);
            dst[c] = w;
          }
        }
      }
      TRP(4);
      ph ^= 1;
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 11) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}


// =====================================================================================================================
// attn_l64_kernel -- Hisfrag model: long sequences (patch tokens a multiple of 256 queries / 128 keys), head_dim 64.
//   Work item = (sequence, head, 256 patch queries): two softmax groups (128 query rows = 4 warps, one thread per row)
//   share one ring of 128-key K/V stages. A group consumes a stage as two 64-key HALF TILES with two score buffers in
//   TMEM: while its threads run the softmax of half tile u (tcgen05.ld -> row max -> ex2 -> packed fp16 P written back
//   over S with tcgen05.st), the tensor pipe executes PV(u-1) and QK^T(u+1), issued earlier by the MMA warp -- the MMA
//   round trip is hidden behind the other buffer's softmax and the group never idles. P feeds the second MMA straight
//   from TMEM (A operand), V is consumed in place as an MN-major operand.
//   Online softmax with a LAZY, per-thread rescale: the running max only moves when a half tile exceeds it by more than
//   2^8; then the thread waits for its group's previous PV, multiplies its own O row in TMEM and carries on.
//   Probabilities are therefore <= 256, exact after the final division by the row sum.
//   The class-token KEY is a last 16-key half tile (row 0 real, the others masked); the class-token QUERY is one extra
//   item per (sequence, head) whose tile has a single live row (group 0 only).
//   Warps: 0-3 group 0, 4-7 group 1, 8 TMA producer, 9 / 10 MMA issuers of group 0 / 1 (warp-uniform code, elected
//   lane; warp 9 also owns the TMEM allocation).
// =====================================================================================================================
struct L64 {
  static constexpr int HD = 64;
  static constexpr int RB = 128;               // bytes per tile row
  static constexpr int QB = 128 * RB;          // one Q tile
  static constexpr int KVB = 128 * RB;         // K (or V) part of a stage: 128 keys
  static constexpr int STAGE = 2 * KVB;        // K, V
  static constexpr int NS = 4;                 // K/V ring depth (stages of 128 keys)
  static constexpr int THREADS = 352;
  static constexpr int GCOLS = 256;            // TMEM columns per group: S/P buffers at +0 and +64, O at +128
  static constexpr int OCOL = 128;
  static constexpr int BAR_BYTES = 512;
  static constexpr int BYTES = 1024 + 4 * QB + NS * STAGE + BAR_BYTES;   // Q double-buffered per group
};

#ifdef VITED_ATTN_TRACE
__device__ unsigned long long g_attn_trace[4 * 128 * 4];   // [who][event index][4 timestamps]; who: 0/1 = MMA warp for group 0/1, 2/3 = softmax warp 0 of group 0/1
#define TR(who, idx, k) do { if (blockIdx.x == 0 && lane == 0 && (idx) < 128) g_attn_trace[((who) * 128 + (idx)) * 4 + (k)] = clock64(); } while (0)
#else
#define TR(who, idx, k) do { } while (0)
#endif

struct L64Maps {
  CUtensorMap q_tile, q_row, k_tile, k_row, v_tile, v_row;   // boxes {64, 128} and {64, 1}, 128B swizzle
};

__global__ void __launch_bounds__(L64::THREADS, 1)
attn_l64_kernel(AttnArgs a, const __grid_constant__ L64Maps maps, int n_items) {
  using C = L64;
  extern __shared__ uint8_t attn_tc_smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(attn_tc_smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sQ = smem;                          // [group][buffer][128 x 128 B]
  uint8_t* sKV = smem + 4 * C::QB;             // [NS][K | V]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sKV + C::NS * C::STAGE);
  uint64_t* kv_full = bars;                    // [NS] TMA bytes landed
  uint64_t* kv_empty = kv_full + C::NS;        // [NS] both groups' PVs on the stage have finished (2 commits / arrivals)
  uint64_t* q_full = kv_empty + C::NS;         // [group*2 + buffer]
  uint64_t* q_empty = q_full + 4;              // [group*2 + buffer] the item's last QK^T has read the Q tile (commit)
  uint64_t* s_full = q_empty + 4;              // [group*2 + buffer] scores of a half tile are in TMEM (commit)
  uint64_t* p_ready = s_full + 4;              // [group*2 + buffer] probabilities are in TMEM (4 warps)
  uint64_t* o_done = p_ready + 4;              // [group*2 + (half tile & 1)] PV of that half tile has finished (commit)
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(o_done + 4);

  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const int H = a.n_heads;
  const int n_qp = a.nq_patch / 256;                         // 256-query blocks per (sequence, head)
  const int per_bh = n_qp + (a.q_has_cls ? 1 : 0);           // + the class-token item
  const int n_kt = a.nk_patch / 128;                         // full 128-key stages per item
  const int n_st = n_kt + (a.k_has_cls ? 1 : 0);             // stages per item (the last one = class-token key)
  const int U = 2 * n_kt + (a.k_has_cls ? 1 : 0);            // half tiles per item
  const int n_my = (n_items - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;

  // stale rows of the ring enter masked score columns / multiply zero probabilities: they only have to be finite
  for (int i = tid; i < (4 * C::QB + C::NS * C::STAGE) / 16; i += C::THREADS)
    reinterpret_cast<uint4*>(smem)[i] = make_uint4(0, 0, 0, 0);
  if (tid == 0) {
    for (int s = 0; s < C::NS; ++s) { mbar_init(&kv_full[s], 1); mbar_init(&kv_empty[s], 2); }
    for (int j = 0; j < 4; ++j) {
      mbar_init(&q_full[j], 1); mbar_init(&q_empty[j], 1); mbar_init(&s_full[j], 1); mbar_init(&p_ready[j], 4);
    }
    for (int j = 0; j < 4; ++j) mbar_init(&o_done[j], 1);
    fence_mbar_init();
    tma_prefetch_desc(&maps.q_tile);
    tma_prefetch_desc(&maps.k_tile);
    tma_prefetch_desc(&maps.v_tile);
  }
  if (warp == 9) {
    tmem_alloc(tmem_holder, 512);
    tmem_relinquish();
  }
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;
  auto is_cls_item = [&](int i) { return (((int)blockIdx.x + i * (int)gridDim.x) % per_bh) == n_qp; };

  if (warp == 8) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int stage = 0;
      uint32_t ph = 0;
      uint32_t qn[2] = {0, 0};      // Q tiles loaded so far per group (buffer = n & 1, phase = (n >> 1) & 1)
      for (int i = 0; i < n_my; ++i) {
        const int item = (int)blockIdx.x + i * (int)gridDim.x;
        const int bh = item / per_bh, qp = item - bh * per_bh;
        const int b = bh / H, h = bh - b * H;
        const int kvb = a.kv_index ? __ldg(a.kv_index + b) : b;
        const int col = h * C::HD;
        const bool cls_item = qp == n_qp;
        for (int g = 0; g < (cls_item ? 1 : 2); ++g) {     // group 1 has no queries in the class-token item
          const int qb = g * 2 + (int)(qn[g] & 1);
          mbar_wait(&q_empty[qb], ((qn[g] >> 1) & 1) ^ 1, 60);
          if (cls_item) {
            mbar_arrive_expect_tx(&q_full[qb], C::RB);
            tma_load_2d(&maps.q_row, &q_full[qb], sQ + qb * C::QB, col, a.n_seq * a.nq_patch + b);
          } else {
            mbar_arrive_expect_tx(&q_full[qb], C::QB);
            tma_load_2d(&maps.q_tile, &q_full[qb], sQ + qb * C::QB, col, b * a.nq_patch + qp * 256 + g * 128);
          }
          ++qn[g];
        }
        for (int t = 0; t < n_st; ++t) {
          mbar_wait(&kv_empty[stage], ph ^ 1, 62);
          uint8_t* st = sKV + stage * C::STAGE;
          if (t < n_kt) {
            mbar_arrive_expect_tx(&kv_full[stage], 2 * C::KVB);
            tma_load_2d(&maps.k_tile, &kv_full[stage], st, col, kvb * a.nk_patch + t * 128);
            tma_load_2d(&maps.v_tile, &kv_full[stage], st + C::KVB, col, kvb * a.nk_patch + t * 128);
          } else {
            mbar_arrive_expect_tx(&kv_full[stage], 2 * C::RB);
            tma_load_2d(&maps.k_row, &kv_full[stage], st, col, a.n_kv_seq * a.nk_patch + kvb);
            tma_load_2d(&maps.v_row, &kv_full[stage], st + C::KVB, col, a.n_kv_seq * a.nk_patch + kvb);
          }
          if (++stage == C::NS) { stage = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp >= 9) {
    // ===================== MMA issuer of group g = warp - 9 (warp-uniform; tcgen05 ops on one elected lane) ==========
    // A lean linear program per item: QK^T(0), QK^T(1), then for every half tile u: PV(u) as soon as P(u) is in TMEM
    // and QK^T(u+2) right behind it into the same score buffer (the tensor pipe runs in issue order). This warp is on
    // the critical path of its group (a single warp executes ~1 dependent instruction per 5 cycles), so it carries
    // no bookkeeping beyond a few counters: an earlier version with one generic cursor-driven warp for both groups
    // spent ~1300 cycles per PV + QK^T pair and starved the softmax warps (tools/trace_attn_l64.py).
    const int g = warp - 9;
    const uint32_t idesc_qk64 = umma_idesc_f16(128, 64), idesc_qk16 = umma_idesc_f16(128, 16);
    const uint32_t idesc_pv = umma_idesc_f16(128, C::HD) | kIdescBMajorMN;
    const uint32_t t_col = tmem_base + g * C::GCOLS;
    const uint32_t kv_base = smem_u32(sKV);
    int stage = 0, qs = 0;          // K/V stage of the next PV / of the next QK^T
    uint32_t kv_ph = 0, qph = 0;
    uint32_t qn = 0, j = 0, pj = 0; // Q tiles consumed, QK^T issued, PV issued
    for (int i = 0; i < n_my; ++i) {
      if (g == 1 && is_cls_item(i)) {
        // no queries for this group in the class-token item: release its K/V stages as they land
        for (int t = 0; t < n_st; ++t) {
          mbar_wait(&kv_full[stage], kv_ph, 65);
          if (elect_one_sync()) mbar_arrive(&kv_empty[stage]);
          __syncwarp();
          if (++stage == C::NS) { stage = 0; kv_ph ^= 1; }
        }
        qs = stage; qph = kv_ph;
        continue;
      }
      const int qb = g * 2 + (int)(qn & 1);
      mbar_wait(&q_full[qb], (qn >> 1) & 1, 66);
      const uint64_t dq = umma_desc_sw128(smem_u32(sQ + qb * C::QB));
      auto issue_qk = [&](int u) {
        if ((u & 1) == 0) mbar_wait(&kv_full[qs], qph, 63);
        tc_fence_after();
        const uint64_t dk = umma_desc_sw128(kv_base + qs * C::STAGE + (u & 1) * (64 * C::RB));
        const uint32_t t_s = t_col + (j & 1) * 64;
        const bool cls_tile = u >= 2 * n_kt, last = u + 1 == U;
        if (elect_one_sync()) {
#pragma unroll
          for (int k = 0; k < C::HD / 16; ++k)
            umma_f16(t_s, dq + 2 * k, dk + 2 * k, cls_tile ? idesc_qk16 : idesc_qk64, k);
          umma_commit(&s_full[g * 2 + (j & 1)]);
          if (last) umma_commit(&q_empty[qb]);
        }
        __syncwarp();
        ++j;
        if ((u & 1) == 1 || last) { if (++qs == C::NS) { qs = 0; qph ^= 1; } }
      };
      issue_qk(0);
      if (U > 1) issue_qk(1);
      for (int u = 0; u < U; ++u) {
        const bool cls_tile = u >= 2 * n_kt;
        const bool stage_done = (u & 1) == 1 || u + 1 == U;
        const uint32_t t_p = t_col + (pj & 1) * 64;
        mbar_wait(&p_ready[g * 2 + (pj & 1)], (pj >> 1) & 1, 64);
        tc_fence_after();
        const uint64_t dv = umma_desc_sw(kv_base + stage * C::STAGE + C::KVB + (u & 1) * (64 * C::RB), 128);
        if (elect_one_sync()) {
          if (cls_tile) {
            umma_f16_ts(t_col + C::OCOL, t_p, dv, idesc_pv, u != 0 ? 1u : 0u);
          } else {
#pragma unroll
            for (int k = 0; k < 4; ++k)   // 16 keys per step = two 8-key groups of 1024 B = +128 in the (addr >> 4) field
              umma_f16_ts(t_col + C::OCOL, t_p + 8 * k, dv + 128 * k, idesc_pv, (u | k) != 0 ? 1u : 0u);
          }
          umma_commit(&o_done[g * 2 + (pj & 1)]);
          if (stage_done) umma_commit(&kv_empty[stage]);
        }
        __syncwarp();
        ++pj;
        if (stage_done) { if (++stage == C::NS) { stage = 0; kv_ph ^= 1; } }
        if (u + 2 < U) issue_qk(u + 2);
      }
      ++qn;
    }
  } else {
    // ===================== softmax group g = warp / 4: one thread per query row =====================
    const int g = warp >> 2, quarter = warp & 3;
    const int row = quarter * 32 + lane;
    const float sl2 = a.scale * kLog2e;
    const uint32_t t_col = tmem_base + g * C::GCOLS;
    const uint32_t t_row = t_col + (static_cast<uint32_t>(quarter * 32) << 16);
    uint32_t j = 0;        // half tiles processed by this group so far (score buffer = j & 1, phase = (j >> 1) & 1)
    // Wait until PV of this group's half tile number jj (and, the tensor pipe being in order, every earlier one) has
    // finished. PV(jj) commits to o_done[parity of jj]; the next commit on the same barrier is PV(jj + 2), which cannot
    // be issued before this thread has published P(jj + 2) -- so the barrier is never more than one phase ahead of the
    // waiter and the parity wait cannot alias. (A single barrier per group can: with both final PVs already complete, a
    // wait for the older parity equals the parity of the current, incomplete phase and never returns.)
    auto wait_pv = [&](uint32_t jj, int tag) { mbar_wait(&o_done[g * 2 + (jj & 1)], (jj >> 1) & 1u, tag); };
    // The running max of some row of this warp moved by more than the threshold: wait for the group's previous PV and
    // rescale the O rows. The decision is taken PER WARP (__any_sync at the call sites) and every lane runs the sequence:
    // tcgen05.ld / st / wait are .sync.aligned, i.e. warp-collective -- executed under a per-thread condition (as this
    // was first written) they hang as soon as a real rescale happens, which random-init weights never trigger and the
    // kernel tests did not reach until test_long_attention_lazy_rescale_paths. Lanes that do not need it multiply by 1.
    auto rescale = [&](bool need, float mt, float& m, float& l) {
      wait_pv(j - 1, 68);
      tc_fence_after();
      const float f = need ? ex2_ftz(m - mt) : 1.f;
      if (need) {
        l *= f;
        m = mt;
      }
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        uint32_t ov[32];
        tmem_ld_32x32b_x32(t_row + C::OCOL + 32 * c, ov);
        tmem_ld_wait();
#pragma unroll
        for (int e = 0; e < 32; ++e) ov[e] = __float_as_uint(__uint_as_float(ov[e]) * f);
        tmem_st_32x32b_x32(t_row + C::OCOL + 32 * c, ov);
      }
    };
    for (int i = 0; i < n_my; ++i) {
      const int item = (int)blockIdx.x + i * (int)gridDim.x;
      const int bh = item / per_bh, qp = item - bh * per_bh;
      const int b = bh / H, h = bh - b * H;
      const bool cls_item = qp == n_qp;
      if (cls_item && g == 1) continue;
      float m = -INFINITY, l = 0.f;
      for (int u = 0; u < U; ++u, ++j) {
        const int sb = g * 2 + (int)(j & 1);
        const uint32_t t_s = t_row + (j & 1) * 64;
        if (quarter == 0) TR(2 + g, j, 0);
        mbar_wait(&s_full[sb], (j >> 1) & 1u, 67);
        if (quarter == 0) TR(2 + g, j, 1);
        tc_fence_after();
        if (u < 2 * n_kt) {
          uint32_t v0[32], v1[32];
          tmem_ld_32x32b_x32(t_s, v0);
          tmem_ld_32x32b_x32(t_s + 32, v1);
          tmem_ld_wait();
          float mx[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) mx[e] = fmaxf(__uint_as_float(v0[e]), __uint_as_float(v1[e]));
#pragma unroll
          for (int c = 4; c < 32; c += 4)
#pragma unroll
            for (int e = 0; e < 4; ++e)
              mx[e] = fmaxf(mx[e], fmaxf(__uint_as_float(v0[c + e]), __uint_as_float(v1[c + e])));
          const float mt = fmaxf(fmaxf(mx[0], mx[1]), fmaxf(mx[2], mx[3])) * sl2;
          if (u == 0) m = mt;
          {
            const bool need = u != 0 && mt > m + 8.f;      // lazy: probabilities stay <= 2^8 otherwise
            if (__any_sync(0xffffffffu, need)) rescale(need, mt, m, l);
          }
          const float mneg = -m;
          float sum[4] = {0.f, 0.f, 0.f, 0.f};
          {
            uint64_t sum2[2] = {0ull, 0ull};
            {
              uint32_t pk[16];
              softmax_exp_pairs<16>(v0, sl2, mneg, pk, sum2);
              tmem_st_32x32b_x16(t_s, pk);
            }
            {
              uint32_t pk[16];
              softmax_exp_pairs<16>(v1, sl2, mneg, pk, sum2);
              tmem_st_32x32b_x16(t_s + 16, pk);
            }
            f2_unpack(sum2[0], sum[0], sum[1]);
            f2_unpack(sum2[1], sum[2], sum[3]);
          }
          l += (sum[0] + sum[1]) + (sum[2] + sum[3]);
        } else {
          // class-token key half tile: column 0 is the only real key
          uint32_t vc[8];
          tmem_ld_32x32b_x8(t_s, vc);
          tmem_ld_wait();
          const float mt = __uint_as_float(vc[0]) * sl2;
          if (u == 0) m = mt;
          {
            const bool need = u != 0 && mt > m + 8.f;
            if (__any_sync(0xffffffffu, need)) rescale(need, mt, m, l);
          }
          const float pc = ex2_ftz(mt - m);
          l += pc;
          uint32_t pc8[8] = {pack_act(pc, 0.f), 0u, 0u, 0u, 0u, 0u, 0u, 0u};
          tmem_st_32x32b_x8(t_s, pc8);
        }
        tmem_st_wait();
        tc_fence_before();
        if (quarter == 0) TR(2 + g, j, 2);
        __syncwarp();
        if (lane == 0) mbar_arrive(&p_ready[sb]);   // 4 warps: P (and any rescaled O row) is in TMEM -> PV may be issued
      }
      // ---- item epilogue: O / l -> fp16 -> global ----
      wait_pv(j - 1, 71);
      tc_fence_after();
      {
        const float inv = 1.f / l;
        size_t orow = 0;
        bool valid;
        if (cls_item) { valid = row == 0; orow = (size_t)a.n_seq * a.nq_patch + b; }
        else { valid = true; orow = (size_t)b * a.nq_patch + qp * 256 + g * 128 + row; }
        uint4* dst = reinterpret_cast<uint4*>(a.o + orow * a.o_ld + h * C::HD);
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          uint32_t ov[32];
          tmem_ld_32x32b_x32(t_row + C::OCOL + 32 * c, ov);
          tmem_ld_wait();
          if (valid) {
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              uint4 w;
              w.x = pack_act(__uint_as_float(ov[8 * e + 0]) * inv, __uint_as_float(ov[8 * e + 1]) * inv);
              w.y = pack_act(__uint_as_float(ov[8 * e + 2]) * inv, __uint_as_float(ov[8 * e + 3]) * inv);
              w.z = pack_act(__uint_as_float(ov[8 * e + 4]) * inv, __uint_as_float(ov[8 * e + 5]) * inv);
              w.w = pack_act(__uint_as_float(ov[8 * e + 6]) * inv, __uint_as_float(ov[8 * e + 7]) * inv);
              dst[4 * c + e] = w;
            }
          }
        }
        tc_fence_before();   // (the next item's first PV overwrites O only after every warp has published its next P)
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 9) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

}  // namespace

// true when the tcgen05 kernel covers this problem (the mma.sync kernel in attention.cu covers everything else)
static bool p64_shape(const AttnArgs& a) { return a.head_dim == 32 && a.nq_patch == 64 && a.nk_patch == 64; }
static bool l64_shape(const AttnArgs& a) {
  return a.head_dim == 64 && a.nq_patch >= 256 && a.nq_patch % 256 == 0 && a.nk_patch >= 128 && a.nk_patch % 128 == 0;
}
bool attention_tc_supported(const AttnArgs& a) { return a.n_heads >= 1 && (p64_shape(a) || l64_shape(a)); }

static int attention_tc_l64(const AttnArgs& a, cudaStream_t stream) {
  const size_t items = (size_t)a.n_seq * a.n_heads * (a.nq_patch / 256 + (a.q_has_cls ? 1 : 0));
  VITED_CHECK(items < ((size_t)1 << 31), "attention_tc: too many work items");
  static PerDeviceOnce once;
  const int sms = device_sm_count();
  if (once.first())
    VITED_CUDA_OK(cudaFuncSetAttribute(attn_l64_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, L64::BYTES));
  const uint64_t cols = (uint64_t)a.n_heads * 64;
  const uint64_t q_rows = (uint64_t)a.n_seq * a.nq_patch + (a.q_has_cls ? a.n_seq : 0);
  const uint64_t k_rows = (uint64_t)a.n_kv_seq * a.nk_patch + (a.k_has_cls ? a.n_kv_seq : 0);
  L64Maps maps;
  if (make_tmap_act_2d(&maps.q_tile, a.q, cols, q_rows, (uint64_t)a.q_ld * 2, 64, 128, 128)) return 1;
  if (make_tmap_act_2d(&maps.q_row, a.q, cols, q_rows, (uint64_t)a.q_ld * 2, 64, 1, 128)) return 1;
  if (make_tmap_act_2d(&maps.k_tile, a.k, cols, k_rows, (uint64_t)a.k_ld * 2, 64, 128, 128)) return 1;
  if (make_tmap_act_2d(&maps.k_row, a.k, cols, k_rows, (uint64_t)a.k_ld * 2, 64, 1, 128)) return 1;
  if (make_tmap_act_2d(&maps.v_tile, a.v, cols, k_rows, (uint64_t)a.v_ld * 2, 64, 128, 128)) return 1;
  if (make_tmap_act_2d(&maps.v_row, a.v, cols, k_rows, (uint64_t)a.v_ld * 2, 64, 1, 128)) return 1;
  const unsigned grid = (unsigned)(items < (size_t)sms ? items : (size_t)sms);
  attn_l64_kernel<<<grid, L64::THREADS, L64::BYTES, stream>>>(a, maps, (int)items);
  VITED_CUDA_OK(cudaGetLastError());
  return 0;
}

static int attention_tc_p64(const AttnArgs& a, cudaStream_t stream) {
  const size_t units = (size_t)a.n_seq * a.n_heads;
  VITED_CHECK(units < ((size_t)1 << 31), "attention_tc: too many work units");
  static PerDeviceOnce once;
  const int sms = device_sm_count();
  if (once.first())
    VITED_CUDA_OK(cudaFuncSetAttribute(attn_p64_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, P64::BYTES));
  const uint64_t cols = (uint64_t)a.n_heads * 32;
  const uint64_t q_rows = (uint64_t)a.n_seq * 64 + (a.q_has_cls ? a.n_seq : 0);
  const uint64_t k_rows = (uint64_t)a.n_kv_seq * 64 + (a.k_has_cls ? a.n_kv_seq : 0);
  P64Maps maps;
  if (make_tmap_act_2d(&maps.q_tile, a.q, cols, q_rows, (uint64_t)a.q_ld * 2, 32, 64, 64)) return 1;
  if (make_tmap_act_2d(&maps.q_row, a.q, cols, q_rows, (uint64_t)a.q_ld * 2, 32, 1, 64)) return 1;
  if (make_tmap_act_2d(&maps.k_tile, a.k, cols, k_rows, (uint64_t)a.k_ld * 2, 32, 64, 64)) return 1;
  if (make_tmap_act_2d(&maps.k_row, a.k, cols, k_rows, (uint64_t)a.k_ld * 2, 32, 1, 64)) return 1;
  if (make_tmap_act_2d(&maps.v_tile, a.v, cols, k_rows, (uint64_t)a.v_ld * 2, 32, 64, 64)) return 1;
  if (make_tmap_act_2d(&maps.v_row, a.v, cols, k_rows, (uint64_t)a.v_ld * 2, 32, 1, 64)) return 1;
  const unsigned grid = (unsigned)(units < (size_t)sms ? units : (size_t)sms);
  attn_p64_kernel<<<grid, P64::THREADS, P64::BYTES, stream>>>(a, maps, (int)units);
  VITED_CUDA_OK(cudaGetLastError());
  return 0;
}

int attention_tc(const AttnArgs& a, cudaStream_t stream) {
  VITED_CHECK(attention_tc_supported(a), "attention_tc: unsupported shape");
  if (l64_shape(a)) return attention_tc_l64(a, stream);
  return attention_tc_p64(a, stream);
}

}  // namespace vited


#ifdef VITED_ATTN_TRACE
extern "C" __attribute__((visibility("default"))) int vited_debug_p64_trace(unsigned long long* out) {
  return (int)cudaMemcpyFromSymbol(out, vited::g_p64_trace, sizeof(unsigned long long) * 4 * 64 * 8);
}
extern "C" __attribute__((visibility("default"))) int vited_debug_attn_trace(unsigned long long* out) {
  return (int)cudaMemcpyFromSymbol(out, vited::g_attn_trace, sizeof(unsigned long long) * 4 * 128 * 4);
}
#endif
