// Self- and cross-attention for the ViT-ED blocks (reference: models/vision_transformer.py:56-80 Attention.forward,
// :174-200 CrossAttention.forward; SDPA default scale head_dim^-0.5, no mask, no dropout at eval).
//
// Flash-style: persistent CTAs, one work item = 64 patch queries of one (sequence, head); Q/K/V tiles arrive by TMA
// (hardware-swizzled boxes, mbarrier ring), softmax statistics stay in registers and are combined with quad shuffles.
// The class token never costs a second 64-row tile: as a query it is row 64 of the Q tile (fifth warp), as a key it
// is a ninth 8-key MMA tile.
//
// Token rows live in the "split" layout: n_seq*n_patch patch rows, then n_seq cls rows.
#include "kernels.h"

namespace vited {

constexpr float kLog2e = 1.4426950408889634f;

// 2^x on the MUFU unit, flush-to-zero (inputs are <= 0 or -inf here); plain exp2f() adds a denormal-range fix-up
// (3-4 extra instructions per element) that this instruction-bound kernel cannot afford.
__device__ __forceinline__ float ex2_ftz(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

template <int HD>
struct AttnSmem {
  static constexpr int RB = HD * 2;              // bytes per tile row (dense; TMA-swizzled 64B / 128B)
  static constexpr int ROWS = 80;                // 64 patch rows + the class-token row (64) + 15 zero rows
  static constexpr int TB = ROWS * RB;           // one tile in bytes (5120 / 10240: a multiple of 1024)
  static constexpr int STAGE = 3 * TB;           // Q, K, V tiles
  static constexpr int NST = 3;                  // TMA ring depth
  static constexpr int OLD = HD + 8;             // padded row (elements) of the per-warp output staging
  static constexpr int OB = ROWS * OLD * 2;
  static constexpr int BYTES = 1024 + NST * STAGE + OB + 64;
};

struct AttnMaps {
  CUtensorMap q_tile, q_row, k_tile, k_row, v_tile, v_row;   // boxes {HD, 64} and {HD, 1}
};

// Persistent flash attention for (sequence, head, 64-query block) work items and 64-key chunks, fed by TMA.
//  * One thread (lane 0 of warp 4) keeps a 3-deep ring of TMA box loads in flight: the 64x{32|64} Q / K / V tiles of
//    the step two ahead land in hardware-swizzled shared memory and complete on an mbarrier, so the five compute warps
//    execute no address arithmetic or copy instructions at all (the cp.async version spent 40 % of its issue slots
//    there; profiles/README.md).
//  * Five identical MMA warps: warps 0-3 own 16 patch queries each; warp 4 owns a 16-row tile whose row 0 is the
//    class-token query (row 64 of the Q tile, rows 65-79 are zeros).
//  * The class-token KEY/VALUE sit in row 64 of the K/V tiles and are consumed as a ninth 8-key MMA tile (first
//    chunk only), so 65-token sequences cost 9/8 of a 64-token one instead of 2x.
//  * cls_only: only warp 4 computes (last decoder layer: only row 0 of each sequence reaches the head).
template <int HD>
__global__ void __launch_bounds__(160, HD == 32 ? 4 : 2) attn_mma_kernel(AttnArgs a, const __grid_constant__ AttnMaps maps, int n_items,
                                                       int cls_only) {
  using SM = AttnSmem<HD>;
  constexpr int RB = SM::RB;
  constexpr int NST = SM::NST;
  constexpr int OLD = SM::OLD;
  constexpr int PIECES = HD / 8;
  extern __shared__ uint8_t attn_smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(attn_smem_raw) + 1023) & ~uintptr_t(1023));
  act_t* sO = reinterpret_cast<act_t*>(smem + NST * SM::STAGE);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + NST * SM::STAGE + SM::OB);
  uint64_t* empty = full + NST;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int qblocks = cls_only ? 1 : (a.nq_patch + 63) / 64;
  const int n_chunks = (a.nk_patch + 63) / 64;
  const bool ragged_k = (a.nk_patch & 63) != 0;
  const float sl2 = a.scale * kLog2e;
  const int g = lane >> 2, t = lane & 3;
  const int mi = lane >> 3, ri = lane & 7;
  const int sw = HD == 32 ? ((ri >> 1) & 3) : ri;   // swizzle term of this lane's ldmatrix rows (row % 8 == ri)

  // rows 65..79 of every tile are never loaded: zero them once (they enter the MMAs as exact zeros)
  for (int i = tid; i < NST * 3 * (15 * RB / 16); i += 160) {
    const int tile = i / (15 * RB / 16), r = i % (15 * RB / 16);
    *reinterpret_cast<uint4*>(smem + tile * SM::TB + 65 * RB + r * 16) = make_uint4(0, 0, 0, 0);
  }
  if (tid == 0) {
    for (int s2 = 0; s2 < NST; ++s2) {
      mbar_init(&full[s2], 1);
      mbar_init(&empty[s2], 5);
    }
    fence_mbar_init();
    tma_prefetch_desc(&maps.q_tile);
    tma_prefetch_desc(&maps.k_tile);
    tma_prefetch_desc(&maps.v_tile);
  }
  fence_proxy_async_smem();   // the generic-proxy zero fill is ordered before later async-proxy (TMA) writes nearby
  __syncthreads();

  // work-item cursor in mixed radix (qb, h, b): stepping by gridDim.x needs no division
  struct Cursor { int item, qb, h, b; };
  const int H = a.n_heads;
  const int step_qb = (int)(gridDim.x % qblocks);
  const int step_h = (int)((gridDim.x / qblocks) % H);
  const int step_b = (int)(gridDim.x / qblocks / H);
  auto advance = [&](Cursor& c) {
    c.item += gridDim.x;
    c.qb += step_qb;
    if (c.qb >= qblocks) { c.qb -= qblocks; c.h += 1; }
    c.h += step_h;
    if (c.h >= H) { c.h -= H; c.b += 1; }
    c.b += step_b;
  };
  Cursor cc;
  cc.item = blockIdx.x;
  cc.qb = (int)(blockIdx.x % qblocks);
  cc.h = (int)((blockIdx.x / qblocks) % H);
  cc.b = (int)(blockIdx.x / qblocks / H);

  // ---- producer state (used by lane 0 of warp 4 only) ----
  Cursor fc = cc;
  int f_kc = 0, f_stage = 0;
  uint32_t f_phase = 0;
  auto produce = [&]() {     // issue the TMA loads of the next not-yet-fetched step (if any)
    if (fc.item >= n_items) return;
    mbar_wait(&empty[f_stage], f_phase ^ 1, 40);
    uint8_t* st = smem + f_stage * SM::STAGE;
    const int kvb = a.kv_index ? __ldg(a.kv_index + fc.b) : fc.b;
    const int col = fc.h * HD;
    uint32_t bytes = 2 * 64 * RB;
    if (f_kc == 0) {
      if (!cls_only) bytes += 64 * RB;
      if (a.q_has_cls && fc.qb == 0) bytes += RB;
      if (a.k_has_cls) bytes += 2 * RB;
    }
    mbar_arrive_expect_tx(&full[f_stage], bytes);
    if (f_kc == 0) {
      if (!cls_only) tma_load_2d(&maps.q_tile, &full[f_stage], st, col, fc.b * a.nq_patch + fc.qb * 64);
      if (a.q_has_cls && fc.qb == 0)
        tma_load_2d(&maps.q_row, &full[f_stage], st + 64 * RB, col, a.n_seq * a.nq_patch + fc.b);
      if (a.k_has_cls) {
        tma_load_2d(&maps.k_row, &full[f_stage], st + SM::TB + 64 * RB, col, a.n_kv_seq * a.nk_patch + kvb);
        tma_load_2d(&maps.v_row, &full[f_stage], st + 2 * SM::TB + 64 * RB, col, a.n_kv_seq * a.nk_patch + kvb);
      }
    }
    tma_load_2d(&maps.k_tile, &full[f_stage], st + SM::TB, col, kvb * a.nk_patch + f_kc * 64);
    tma_load_2d(&maps.v_tile, &full[f_stage], st + 2 * SM::TB, col, kvb * a.nk_patch + f_kc * 64);
    if (++f_kc == n_chunks) { f_kc = 0; advance(fc); }
    if (++f_stage == NST) { f_stage = 0; f_phase ^= 1; }
  };
  const bool is_producer = (warp == 4 && lane == 0);
  if (is_producer) {
#pragma unroll
    for (int i = 0; i < NST - 1; ++i) produce();
  }

  // ---- per-warp state (lives across the chunks of one item) ----
  uint32_t qf[HD / 16][4];
  float o_acc[HD / 8][4];
  float m_row[2], l_row[2];

  int kc = 0, stage = 0;
  uint32_t phase = 0;
  while (cc.item < n_items) {
    if (is_producer) produce();
    __syncwarp();
    mbar_wait(&full[stage], phase, 41);

    const uint32_t sQ = smem_u32(smem + stage * SM::STAGE);
    const uint32_t sK = sQ + SM::TB;
    const uint32_t sV = sQ + 2 * SM::TB;
    const int qb = cc.qb;
    const bool active = warp == 4 ? (a.q_has_cls && qb == 0) : !cls_only;

    if (active) {
      if (kc == 0) {
#pragma unroll
        for (int ks = 0; ks < HD / 16; ++ks) {
          const int row = warp * 16 + (mi & 1) * 8 + ri;
          const int c16 = ks * 2 + (mi >> 1);
          ldsm_x4(sQ + row * RB + ((c16 ^ sw) << 4), qf[ks][0], qf[ks][1], qf[ks][2], qf[ks][3]);
        }
        m_row[0] = m_row[1] = -INFINITY;
        l_row[0] = l_row[1] = 0.f;
#pragma unroll
        for (int nt = 0; nt < HD / 8; ++nt) o_acc[nt][0] = o_acc[nt][1] = o_acc[nt][2] = o_acc[nt][3] = 0.f;
      }
      const bool with_cls_key = a.k_has_cls && kc == 0;   // ninth key tile: row 64 = class-token key

      // ---- S = Q K^T : 16 queries x (64 [+8]) keys per warp, raw (unscaled) scores ----
      float s[9][4];
#pragma unroll
      for (int nt = 0; nt < 9; ++nt) s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f;
#pragma unroll
      for (int np = 0; np < 4; ++np) {
#pragma unroll
        for (int ks = 0; ks < HD / 16; ++ks) {
          const int key = np * 16 + (mi >> 1) * 8 + ri;
          const int c16 = ks * 2 + (mi & 1);
          uint32_t b0, b1, b2, b3;
          ldsm_x4(sK + key * RB + ((c16 ^ sw) << 4), b0, b1, b2, b3);
          mma_f16_16816(s[2 * np], qf[ks], b0, b1);
          mma_f16_16816(s[2 * np + 1], qf[ks], b2, b3);
        }
      }
      if (with_cls_key) {
#pragma unroll
        for (int ks = 0; ks < HD / 16; ks += 2) {
          // one ldmatrix.x4 = the (keys 64..71) B fragments of two k-steps
          const int c16 = ks * 2 + mi;
          uint32_t b0, b1, b2, b3;
          ldsm_x4(sK + (64 + ri) * RB + ((c16 ^ sw) << 4), b0, b1, b2, b3);
          mma_f16_16816(s[8], qf[ks], b0, b1);
          mma_f16_16816(s[8], qf[ks + 1], b2, b3);
        }
      }
      // ---- online softmax (rows g and g+8 of this warp's tile) ----
      if (ragged_k) {
        const int k0 = kc * 64;
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
          const int key = k0 + nt * 8 + 2 * t;
          if (key >= a.nk_patch) s[nt][0] = s[nt][2] = -INFINITY;
          if (key + 1 >= a.nk_patch) s[nt][1] = s[nt][3] = -INFINITY;
        }
      }
      // only key 64 of the ninth tile exists (thread t == 0, first element)
      if (!(with_cls_key && t == 0)) s[8][0] = s[8][2] = -INFINITY;
      s[8][1] = s[8][3] = -INFINITY;
      float mx0 = fmaxf(s[8][0], s[8][1]), mx1 = fmaxf(s[8][2], s[8][3]);
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        mx0 = fmaxf(mx0, fmaxf(s[nt][0], s[nt][1]));
        mx1 = fmaxf(mx1, fmaxf(s[nt][2], s[nt][3]));
      }
      mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1)); mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
      mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1)); mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
      const float mn0 = fmaxf(m_row[0], mx0 * sl2), mn1 = fmaxf(m_row[1], mx1 * sl2);   // scaled (log2) units
      const float c0 = ex2_ftz(m_row[0] - mn0), c1 = ex2_ftz(m_row[1] - mn1);
      m_row[0] = mn0; m_row[1] = mn1;
      float rs0 = 0.f, rs1 = 0.f;
#pragma unroll
      for (int nt = 0; nt < 9; ++nt) {
        s[nt][0] = ex2_ftz(fmaf(s[nt][0], sl2, -mn0)); s[nt][1] = ex2_ftz(fmaf(s[nt][1], sl2, -mn0));
        s[nt][2] = ex2_ftz(fmaf(s[nt][2], sl2, -mn1)); s[nt][3] = ex2_ftz(fmaf(s[nt][3], sl2, -mn1));
        rs0 += s[nt][0] + s[nt][1];
        rs1 += s[nt][2] + s[nt][3];
      }
      l_row[0] = l_row[0] * c0 + rs0;    // thread-partial row sums; the quad is reduced at the end
      l_row[1] = l_row[1] * c1 + rs1;
      if (kc > 0) {
#pragma unroll
        for (int nt = 0; nt < HD / 8; ++nt) {
          o_acc[nt][0] *= c0; o_acc[nt][1] *= c0;
          o_acc[nt][2] *= c1; o_acc[nt][3] *= c1;
        }
      }
      // ---- O += P V ----
#pragma unroll
      for (int k2 = 0; k2 < 4; ++k2) {
        uint32_t pa[4];
        pa[0] = pack_act(s[2 * k2][0], s[2 * k2][1]);
        pa[1] = pack_act(s[2 * k2][2], s[2 * k2][3]);
        pa[2] = pack_act(s[2 * k2 + 1][0], s[2 * k2 + 1][1]);
        pa[3] = pack_act(s[2 * k2 + 1][2], s[2 * k2 + 1][3]);
#pragma unroll
        for (int dp = 0; dp < HD / 16; ++dp) {
          const int key = k2 * 16 + (mi & 1) * 8 + ri;
          const int c16 = dp * 2 + (mi >> 1);
          uint32_t b0, b1, b2, b3;
          ldsm_x4_trans(sV + key * RB + ((c16 ^ sw) << 4), b0, b1, b2, b3);
          mma_f16_16816(o_acc[2 * dp], pa, b0, b1);
          mma_f16_16816(o_acc[2 * dp + 1], pa, b2, b3);
        }
      }
      if (with_cls_key) {
        // fifth k-step: keys 64..79 (64 = class token, 65..79 are zero rows with zero probabilities)
        uint32_t pa[4];
        pa[0] = pack_act(s[8][0], s[8][1]);
        pa[1] = pack_act(s[8][2], s[8][3]);
        pa[2] = 0u;
        pa[3] = 0u;
#pragma unroll
        for (int dp = 0; dp < HD / 16; ++dp) {
          const int key = 64 + (mi & 1) * 8 + ri;
          const int c16 = dp * 2 + (mi >> 1);
          uint32_t b0, b1, b2, b3;
          ldsm_x4_trans(sV + key * RB + ((c16 ^ sw) << 4), b0, b1, b2, b3);
          mma_f16_16816(o_acc[2 * dp], pa, b0, b1);
          mma_f16_16816(o_acc[2 * dp + 1], pa, b2, b3);
        }
      }
    }
    // this warp is done reading the stage: hand it back to the producer
    __syncwarp();
    if (lane == 0) mbar_arrive(&empty[stage]);

    // ---- finalize the item after its last chunk ----
    if (active && kc == n_chunks - 1) {
      const int h = cc.h;
      const int b = cc.b;
      const int q0 = qb * 64;
      float l0 = l_row[0], l1 = l_row[1];
      l0 += __shfl_xor_sync(0xffffffffu, l0, 1); l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
      l1 += __shfl_xor_sync(0xffffffffu, l1, 1); l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
      const float i0 = 1.f / l0, i1 = 1.f / l1;
      // each warp stages and stores its own 16 rows (only this warp ever touches these sO rows)
#pragma unroll
      for (int nt = 0; nt < HD / 8; ++nt) {
        *reinterpret_cast<uint32_t*>(&sO[(warp * 16 + g) * OLD + nt * 8 + 2 * t]) =
            pack_act(o_acc[nt][0] * i0, o_acc[nt][1] * i0);
        *reinterpret_cast<uint32_t*>(&sO[(warp * 16 + g + 8) * OLD + nt * 8 + 2 * t]) =
            pack_act(o_acc[nt][2] * i1, o_acc[nt][3] * i1);
      }
      __syncwarp();
      if (warp < 4) {
        act_t* obase = a.o + ((size_t)b * a.nq_patch + q0) * a.o_ld + h * HD;
        for (int idx = lane; idx < 16 * PIECES; idx += 32) {
          const int row = warp * 16 + idx / PIECES, pc = idx % PIECES;
          if (q0 + row < a.nq_patch)
            *reinterpret_cast<uint4*>(obase + (size_t)row * a.o_ld + pc * 8) =
                *reinterpret_cast<const uint4*>(&sO[row * OLD + pc * 8]);
        }
      } else if (lane < PIECES) {
        const size_t orow = (size_t)a.n_seq * a.nq_patch + b;   // class-token output row
        *reinterpret_cast<uint4*>(a.o + orow * a.o_ld + h * HD + lane * 8) =
            *reinterpret_cast<const uint4*>(&sO[64 * OLD + lane * 8]);
      }
      __syncwarp();
    }
    if (++kc == n_chunks) { kc = 0; advance(cc); }
    if (++stage == NST) { stage = 0; phase ^= 1; }
  }
}

// ------------------------------------------------------------------------------------------------------------
// debugging reference: one thread per query token, fp32 FMAs, keys streamed through shared memory.
// ------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ size_t tok_row(int n_seq_total, int n_patch, int has_cls, int b, int s) {
  if (has_cls) return s == 0 ? (size_t)n_seq_total * n_patch + b : (size_t)b * n_patch + (s - 1);
  return (size_t)b * n_patch + s;
}

template <int HD>
__global__ void __launch_bounds__(128) attn_simt_kernel(AttnArgs a) {
  __shared__ float Ks[32][HD];
  __shared__ float Vs[32][HD];
  const int nq = a.nq_patch + a.q_has_cls, nk = a.nk_patch + a.k_has_cls;
  const int qblocks = (nq + 127) / 128;
  const int b = blockIdx.x / qblocks, qb = blockIdx.x % qblocks;
  const int h = blockIdx.y;
  const int kvb = a.kv_index ? a.kv_index[b] : b;
  const int sq = qb * 128 + threadIdx.x;
  const bool valid = sq < nq;
  float q[HD], o[HD];
  float m = -INFINITY, l = 0.f;
  if (valid) {
    const size_t row = tok_row(a.n_seq, a.nq_patch, a.q_has_cls, b, sq);
#pragma unroll
    for (int d = 0; d < HD; ++d) q[d] = act2f(a.q[row * a.q_ld + h * HD + d]);
  }
#pragma unroll
  for (int d = 0; d < HD; ++d) o[d] = 0.f;
  for (int k0 = 0; k0 < nk; k0 += 32) {
    __syncthreads();
    for (int idx = threadIdx.x; idx < 32 * HD; idx += 128) {
      const int kk = idx / HD, d = idx % HD;
      float kv = 0.f, vv = 0.f;
      if (k0 + kk < nk) {
        const size_t row = tok_row(a.n_kv_seq, a.nk_patch, a.k_has_cls, kvb, k0 + kk);
        kv = act2f(a.k[row * a.k_ld + h * HD + d]);
        vv = act2f(a.v[row * a.v_ld + h * HD + d]);
      }
      Ks[kk][d] = kv;
      Vs[kk][d] = vv;
    }
    __syncthreads();
    if (valid) {
      const int kmax = min(32, nk - k0);
      for (int kk = 0; kk < kmax; ++kk) {
        float s = 0.f;
#pragma unroll
        for (int d = 0; d < HD; ++d) s += q[d] * Ks[kk][d];
        s *= a.scale;
        const float mn = fmaxf(m, s);
        const float corr = __expf(m - mn);
        const float p = __expf(s - mn);
        l = l * corr + p;
#pragma unroll
        for (int d = 0; d < HD; ++d) o[d] = o[d] * corr + p * Vs[kk][d];
        m = mn;
      }
    }
  }
  if (valid) {
    const size_t row = tok_row(a.n_seq, a.nq_patch, a.q_has_cls, b, sq);
    const float inv = 1.f / l;
#pragma unroll
    for (int d = 0; d < HD; ++d) a.o[row * a.o_ld + h * HD + d] = f2act(o[d] * inv);
  }
}

static int attention_launch(const AttnArgs& a, int cls_only, cudaStream_t stream);

// ---------------------------------------------------------------------------------------------------------------------
// Class-token query only, puzzle shape (head_dim 32, 64 patch keys [+ class-token key]): the pruned last decoder layer.
// One query row per (sequence, head) is 4 KB of K and 4 KB of V against 8 KFLOP -- pure streaming, and the tile
// kernels keep only four such units in flight per SM (0.36 ms per chunk at 2.2 TB/s). Here: one warp per unit, every
// lane owns 8 dims of 8(+1) key rows (row 8 i + lane / 4, dims 8 (lane % 4) ..), all 18 16-byte loads of a unit are
// independent, scores are reduced over the 4 lanes of a row, the softmax runs in fp32 registers, and P.V needs no
// shuffles for P (a lane multiplies the V chunk of the rows whose probability it already holds).
// ---------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void unpack8(const uint4& u, float (&f)[8]) {
  const float2 a = unpack_act(u.x), b = unpack_act(u.y), c = unpack_act(u.z), d = unpack_act(u.w);
  f[0] = a.x; f[1] = a.y; f[2] = b.x; f[3] = b.y; f[4] = c.x; f[5] = c.y; f[6] = d.x; f[7] = d.y;
}

__global__ void __launch_bounds__(256) attn_cls_warp_kernel(AttnArgs a) {
  const int lane = threadIdx.x & 31, sub = lane & 3, rsub = lane >> 2;
  const int n_units = a.n_seq * a.n_heads;
  const int warps = (gridDim.x * blockDim.x) >> 5;
  const float sl2 = a.scale * 1.4426950408889634f;
  for (int unit = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; unit < n_units; unit += warps) {
    const int b = unit / a.n_heads, h = unit - b * a.n_heads;
    const int kvb = a.kv_index != nullptr ? __ldg(a.kv_index + b) : b;
    const size_t col = (size_t)h * 32 + 8 * sub;
    const uint4 qv = __ldg(reinterpret_cast<const uint4*>(a.q + ((size_t)a.n_seq * 64 + b) * a.q_ld + col));
    uint4 kk[9], vv[9];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const size_t r = (size_t)kvb * 64 + 8 * i + rsub;
      kk[i] = __ldg(reinterpret_cast<const uint4*>(a.k + r * a.k_ld + col));
      vv[i] = __ldg(reinterpret_cast<const uint4*>(a.v + r * a.v_ld + col));
    }
    const bool has_c = a.k_has_cls && rsub == 0;               // the class-token key: lanes 0..3
    kk[8] = vv[8] = make_uint4(0, 0, 0, 0);
    if (has_c) {
      const size_t r = (size_t)a.n_kv_seq * 64 + kvb;
      kk[8] = __ldg(reinterpret_cast<const uint4*>(a.k + r * a.k_ld + col));
      vv[8] = __ldg(reinterpret_cast<const uint4*>(a.v + r * a.v_ld + col));
    }
    float q[8];
    unpack8(qv, q);
    float sc[9];
    float mx = -INFINITY;
#pragma unroll
    for (int i = 0; i < 9; ++i) {
      float k8[8];
      unpack8(kk[i], k8);
      float d = 0.f;
#pragma unroll
      for (int e = 0; e < 8; ++e) d = fmaf(q[e], k8[e], d);
      d += __shfl_xor_sync(0xffffffffu, d, 1);
      d += __shfl_xor_sync(0xffffffffu, d, 2);
      sc[i] = (i < 8 || has_c) ? d * sl2 : -INFINITY;
      mx = fmaxf(mx, sc[i]);
    }
#pragma unroll
    for (int o = 4; o < 32; o <<= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    float l = 0.f, acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int i = 0; i < 9; ++i) {
      const float p = exp2f(sc[i] - mx);                        // exp2f(-inf) = 0 for the rows that do not exist
      l += p;
      float v8[8];
      unpack8(vv[i], v8);
#pragma unroll
      for (int e = 0; e < 8; ++e) acc[e] = fmaf(p, v8[e], acc[e]);
    }
#pragma unroll
    for (int o = 4; o < 32; o <<= 1) {
      l += __shfl_xor_sync(0xffffffffu, l, o);
#pragma unroll
      for (int e = 0; e < 8; ++e) acc[e] += __shfl_xor_sync(0xffffffffu, acc[e], o);
    }
    if (rsub == 0) {                                            // lanes 0..3 hold the 32 output dims
      const float inv = 1.f / l;
      uint4 w;
      w.x = pack_act(acc[0] * inv, acc[1] * inv);
      w.y = pack_act(acc[2] * inv, acc[3] * inv);
      w.z = pack_act(acc[4] * inv, acc[5] * inv);
      w.w = pack_act(acc[6] * inv, acc[7] * inv);
      *reinterpret_cast<uint4*>(a.o + ((size_t)a.n_seq * 64 + b) * a.o_ld + col) = w;
    }
  }
}

static bool attn_cls_warp_supported(const AttnArgs& a) {
  return a.head_dim == 32 && a.nq_patch == 64 && a.nk_patch == 64 && a.q_has_cls &&
         a.q_ld % 8 == 0 && a.k_ld % 8 == 0 && a.v_ld % 8 == 0 && a.o_ld % 8 == 0;
}

// class-token query only (last decoder layer): same kernel, only the fifth warp computes.
int attention_cls(const AttnArgs& a, cudaStream_t stream) {
  VITED_CHECK(a.head_dim == 32 || a.head_dim == 64, "attention_cls: head_dim %d not supported (32 or 64)", a.head_dim);
  VITED_CHECK(a.q_has_cls, "attention_cls: the query sequences have no class token");
  if (a.n_seq == 0) return 0;
  if (attn_cls_warp_supported(a)) {
    const int units = a.n_seq * a.n_heads;
    int blocks = (units + 7) / 8;
    if (blocks > 148 * 8) blocks = 148 * 8;
    attn_cls_warp_kernel<<<blocks, 256, 0, stream>>>(a);
    VITED_CUDA_OK(cudaGetLastError());
    return 0;
  }
  return attention_launch(a, 1, stream);
}

int attention(const AttnArgs& a, int impl, cudaStream_t stream) {
  VITED_CHECK(a.head_dim == 32 || a.head_dim == 64, "attention: head_dim %d not supported (32 or 64)", a.head_dim);
  VITED_CHECK(a.q_ld % 8 == 0 && a.k_ld % 8 == 0 && a.v_ld % 8 == 0 && a.o_ld % 8 == 0,
              "attention: row strides must be multiples of 8 elements");
  VITED_CHECK(a.nq_patch > 0 && a.nk_patch > 0, "attention: empty sequences");
  if (a.n_seq == 0) return 0;
  if (impl == IMPL_REF) {
    const int nq = a.nq_patch + a.q_has_cls;
    dim3 grid((unsigned)((size_t)a.n_seq * ((nq + 127) / 128)), a.n_heads);
    if (a.head_dim == 32) attn_simt_kernel<32><<<grid, 128, 0, stream>>>(a);
    else attn_simt_kernel<64><<<grid, 128, 0, stream>>>(a);
  } else {
    if (impl == IMPL_FAST && attention_tc_supported(a)) return attention_tc(a, stream);
    return attention_launch(a, 0, stream);
  }
  VITED_CUDA_OK(cudaGetLastError());
  return 0;
}

static int attention_launch(const AttnArgs& a, int cls_only, cudaStream_t stream) {
  const size_t items = (size_t)a.n_seq * a.n_heads * (cls_only ? 1 : (a.nq_patch + 63) / 64);
  VITED_CHECK(items < (size_t)1 << 31, "attention: too many work items");
  static int per_sm32 = 0, per_sm64 = 0;   // resident CTAs per SM (registers / shared memory; same on every B200)
  static PerDeviceOnce once;
  const int sms = device_sm_count();
  if (once.first()) {
    VITED_CUDA_OK(cudaFuncSetAttribute(attn_mma_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, AttnSmem<32>::BYTES));
    VITED_CUDA_OK(cudaFuncSetAttribute(attn_mma_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, AttnSmem<64>::BYTES));
    VITED_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm32, attn_mma_kernel<32>, 160, AttnSmem<32>::BYTES));
    VITED_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm64, attn_mma_kernel<64>, 160, AttnSmem<64>::BYTES));
    if (per_sm32 < 1) per_sm32 = 1;
    if (per_sm64 < 1) per_sm64 = 1;
  }
  const int per_sm = a.head_dim == 32 ? per_sm32 : per_sm64;
  size_t grid = (size_t)sms * per_sm;
  if (grid > items) grid = items;
  // TMA descriptors: 64-row tiles and single rows (class token) of the q / k / v buffers, hardware swizzle = row bytes
  const int HD = a.head_dim, swz = HD * 2;
  const uint64_t cols = (uint64_t)a.n_heads * HD;
  const uint64_t q_rows = (uint64_t)a.n_seq * a.nq_patch + (a.q_has_cls ? a.n_seq : 0);
  const uint64_t k_rows = (uint64_t)a.n_kv_seq * a.nk_patch + (a.k_has_cls ? a.n_kv_seq : 0);
  AttnMaps maps;
  if (make_tmap_act_2d(&maps.q_tile, a.q, cols, q_rows, (uint64_t)a.q_ld * 2, HD, 64, swz)) return 1;
  if (make_tmap_act_2d(&maps.q_row, a.q, cols, q_rows, (uint64_t)a.q_ld * 2, HD, 1, swz)) return 1;
  if (make_tmap_act_2d(&maps.k_tile, a.k, cols, k_rows, (uint64_t)a.k_ld * 2, HD, 64, swz)) return 1;
  if (make_tmap_act_2d(&maps.k_row, a.k, cols, k_rows, (uint64_t)a.k_ld * 2, HD, 1, swz)) return 1;
  if (make_tmap_act_2d(&maps.v_tile, a.v, cols, k_rows, (uint64_t)a.v_ld * 2, HD, 64, swz)) return 1;
  if (make_tmap_act_2d(&maps.v_row, a.v, cols, k_rows, (uint64_t)a.v_ld * 2, HD, 1, swz)) return 1;
  if (a.head_dim == 32)
    attn_mma_kernel<32><<<(unsigned)grid, 160, AttnSmem<32>::BYTES, stream>>>(a, maps, (int)items, cls_only);
  else
    attn_mma_kernel<64><<<(unsigned)grid, 160, AttnSmem<64>::BYTES, stream>>>(a, maps, (int)items, cls_only);
  VITED_CUDA_OK(cudaGetLastError());
  return 0;
}

}  // namespace vited
