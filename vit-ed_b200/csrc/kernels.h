// Internal launcher interface between the engine (engine.cu) and the kernels. Everything takes raw device
// pointers and a cudaStream_t; every launcher returns 0 on success and sets vited::set_error() otherwise.
#pragma once
#include "common.cuh"

namespace vited {

enum { ACT_NONE = 0, ACT_GELU = 1 };
enum { IMPL_FAST = 0, IMPL_REF = 1, IMPL_MMA_SYNC = 2 };  // IMPL_REF: plain SIMT debugging kernels; IMPL_MMA_SYNC (attention
                                                        // only): force the general mma.sync kernel even where a tcgen05 one exists

// ---- GEMM: C[M,N] (fp16) = act(A[M,K] (fp16, row-major) * W[N,K]^T (fp16, row-major) + bias[N] (f32)) ----
// IMPL_FAST: persistent warp-specialised tcgen05/TMEM kernel fed by TMA (gemm_tc.cu).
int gemm_act(const act_t* A, const act_t* W, const float* bias, act_t* C, int M, int N, int K, int act, int impl,
              cudaStream_t stream);
int gemm_num_sms();
// 2-D fp16 TMA descriptor (driver entry point resolved in gemm_tc.cu); swizzle_bytes in {0, 64, 128}
int make_tmap_act_2d(CUtensorMap* tm, const void* ptr, uint64_t cols, uint64_t rows, uint64_t row_stride_bytes,
                      uint32_t box_cols, uint32_t box_rows, int swizzle_bytes);

int make_tmap_f32_2d(CUtensorMap* tm, const void* ptr, uint64_t cols, uint64_t rows, uint64_t row_stride_bytes,
                     uint32_t box_cols, uint32_t box_rows, int swizzle_bytes);

// ---- fused GEMM + residual + LayerNorm (gemm_ln.cu) ----
//   x[M,384] (f32, in place) += A[M,K] (fp16) * W[384,K]^T (fp16) + bias;  h[M,384] (fp16) = LayerNorm(x) * ln_w + ln_b
// i.e. `x = x + proj(...)` followed by the next `normX(x)` (vision_transformer.py:124-127, :268-272) in ONE kernel: the
// accumulator row never leaves the SM before it is normalised. Only N = 384 (the models' embed_dim) and large M.
bool gemm_resid_ln_supported(int M, int N, int K);
int gemm_resid_ln(const act_t* A, const act_t* W, const float* bias, float* x, const float* ln_w, const float* ln_b,
                  act_t* h, int M, int N, int K, float eps, cudaStream_t stream);

// ---- fused MLP sub-block + residual + LayerNorm (mlp_ln.cu) ----
//   x[M,384] (f32, in place) += GELU(h_in[M,384] W1[hidden,384]^T + b1) W2[384,hidden]^T + b2;  h_out = LayerNorm(x) * ln_w + ln_b
// i.e. `x = x + mlp(norm2(x))` followed by the next layer's `norm1(x)` (vision_transformer.py:126-127, :272) in ONE kernel:
// the [M, hidden] activations never leave the SM. h_out may alias h_in. Only embed_dim 384, hidden a multiple of 64.
bool mlp_resid_ln_supported(int M, int D, int hidden);
int mlp_resid_ln(const act_t* h_in, const act_t* W1, const float* b1, const act_t* W2, const float* b2, float* x,
                 const float* ln_w, const float* ln_b, act_t* h_out, int M, int D, int hidden, float eps,
                 cudaStream_t stream);
// the cross-attention projection + residual + norm2 in front of the same kernel (a decoder CrossBlock's
// `x = x + cross_attn.proj(o); x = x + mlp(norm2(x))` followed by the next layer's norm1):
//   x_mid = x + o[M,384] Wp[384,384]^T + bp;  x = x_mid + fc2(GELU(fc1(LayerNorm(x_mid) * ln2_w + ln2_b)));
//   h_out = LayerNorm(x) * ln_w + ln_b.  x_mid and norm2(x_mid) never leave the SM; x holds the final rows only.
bool cproj_mlp_resid_ln_supported(int M, int D, int K, int hidden);
int cproj_mlp_resid_ln(const act_t* o, const act_t* Wp, const float* bp, float* x, const float* ln2_w,
                       const float* ln2_b, const act_t* W1, const float* b1, const act_t* W2, const float* b2,
                       const float* ln_w, const float* ln_b, act_t* h_out, int M, int D, int hidden, float eps,
                       cudaStream_t stream);

// ---- row-wise kernels (rowops.cu) ----
// x[r,:] = (gather ? src[map(r),:] : x[r,:]) + delta[r,:]; optionally h[r,:] = LayerNorm(x[r,:]) * w + b (fp16).
// Row space is the "split" layout: n_seq*n_patch patch rows followed by n_cls cls rows (n_cls = n_seq or 0).
struct ResidLnArgs {
  float* x;              // [R, D] residual stream (fp32), updated in place when write_x
  const act_t* delta;     // [R, D] or null
  const float* gather_src;   // split-layout source [n_src_seq*n_patch (+ n_src_seq cls rows), D] or null
  const int* gather_idx;     // [n_seq] source item of every destination sequence; source sequence = item - gather_off
  int gather_off;            // first item held in gather_src (vited_score_grid keeps only the columns a row shard needs)
  int n_src_seq;
  const float* ln_w;     // null -> no LayerNorm output
  const float* ln_b;
  act_t* h;               // [R, D]
  int n_seq, n_patch, has_cls, D;
  int write_x;
  float eps;
};
int resid_ln(const ResidLnArgs& a, cudaStream_t stream);

// images [B,3,S,S] f32 -> patch matrix [B*G*G, 3*p*p] fp16, column = c*p*p + py*p + px (Conv2d weight.view order).
// items (device, [B]) non-null: output image b is read from images[items[b]] (a gathered batch, no staging copy).
int im2col_patches(const float* images, act_t* out, int B, int C, int S, int p, cudaStream_t stream,
                   const int* items = nullptr);
// images [B,S,S,C] u8 (HWC bytes) -> the same patch matrix, bit-identical to normalize_u8 + im2col_patches
// (ToTensor + Normalize(.5, .5) folded in). Built for C = 3 and p in {4, 8, 16, 32}; anything else is an error.
int im2col_u8_patches(const uint8_t* images, act_t* out, int B, int C, int S, int p, cudaStream_t stream,
                      const int* items = nullptr);

// x0 (f32, split layout, B sequences): patch rows = tok (fp16 [B*Np, D]) + pos[1+t]; cls rows = cls + pos[0]
int assemble_tokens(const act_t* tok, const float* pos_embed, const float* cls_token, float* x, int B, int n_patch,
                    int D, int with_cls, cudaStream_t stream);

// final: y = LayerNorm(x_cls + delta_cls); logits = y * Wh^T + bh; scattered into the score matrix.
struct HeadArgs {
  const float* x;       // cls rows [P, D] f32
  const act_t* delta;    // cls rows [P, D] or null
  const float* ln_w;
  const float* ln_b;
  const float* head_w;  // [C, D]
  const float* head_b;  // [C]
  float* out;
  const int* ci;        // pair -> ctx item (row of the grid); null => linear output out[p*C + c]
  const int* xj;        // pair -> x2 item (column)
  const int* out_pos;   // non-null: out[out_pos[p]*C + c] (vited_score_pairs: the pair's position in the caller's list)
  int row_begin, n_items;
  int P, D, C;
  float eps;
};
int head_logits(const HeadArgs& a, cudaStream_t stream);

// pair list of grid rows [r0, r1) x column window [ca, cb) on the device, i-major with j ascending:
// ci[p] = i - r0 (context row inside the block), xj[p] = j (absolute item index).
//   mode 0: ordered off-diagonal pairs, j in [ca, cb) \ {i}  (data/datasets/pieces_dataset.py:27-32)
//   mode 1: upper triangle incl. diagonal, j in [max(i, ca), cb)  (hisfrag.py:166-167)
//   mode 2: identity, ci[p] = xj[p] = p for p in [0, r1 - r0)  (two-phase / one-shot decode of B pairs; window unused)
// The whole grid row is the window [0, N). pair_list_count returns the number of pairs (the caller sizes ci / xj with it).
__host__ __device__ size_t pair_list_count(int mode, int r0, int r1, int ca, int cb);
int pair_list(int mode, int r0, int r1, int ca, int cb, int* ci, int* xj, cudaStream_t stream);

// ---- caller-given pair lists (pair_lists.cu): the index work of vited_score_pairs ----
// info block copied back to the host once per call: the header below, then PL_CELLS + k = first sorted position of cell
// k (k <= cells, the last entry = number of valid pairs)
enum { PL_N_BAD = 0, PL_FIRST_BAD, PL_BAD_A, PL_BAD_B, PL_N_CTX, PL_N_X2, PL_CELLS };
// pairs [P, 2] (context item, decoder item); used [2N] zeroed: used[a] / used[N + b] = 1 for valid pairs; invalid ones
// counted in info[PL_N_BAD], the lowest such pair index in info[PL_FIRST_BAD] (preset to 0xffffffff)
int pairs_mark(const int* pairs, int P, int N, int* used, int* info, cudaStream_t stream);
// exclusive prefix sum of n ints (one block; out may alias in); *total = sum (device)
int exclusive_scan(const int* in, int* out, int64_t n, int* total, cudaStream_t stream);
// items[half*N + slot[half*N + i]] = i for the used items of both halves (ascending lists of distinct items)
int pairs_compact(const int* used, const int* slot, int* items, int N, cudaStream_t stream);
// cell of a pair = (context slot / rb) * nw + decoder slot / cw; the sort runs on tiles of T pairs, one warp each
struct PairCells { int rb, cw, nw, T, tiles; };
// hist [cells * tiles] zeroed -> pairs per (cell, tile)
int pairs_bucket_count(const int* pairs, int P, int N, const int* slot, const PairCells& c, int* hist,
                       cudaStream_t stream);
// info[PL_CELLS + k] = hist[k * tiles] (hist exclusive-scanned) and the offending pair's indices, if any
int pairs_cell_starts(const int* pairs, const int* hist, int tiles, int cells, int* info, cudaStream_t stream);
// stable scatter by cell: ci = context slot % rb, xj = decoder slot, out_pos = input position (hist advanced)
int pairs_bucket_scatter(const int* pairs, int P, int N, const int* slot, const PairCells& c, int* hist, int* ci,
                         int* xj, int* out_pos, cudaStream_t stream);

// plain copy/convert helpers
int f32_to_act(const float* in, act_t* out, size_t n, cudaStream_t stream);
int add_delta_out(const float* x, const act_t* delta, float* out, size_t rows, int D, cudaStream_t stream);

// ---- on-device piece preparation (piece_prep.cu): see include/vited_b200.h vited_prepare_pieces ----
int prepare_pieces(const uint8_t* lab, int H, int W, int piece_width, int side, int off, int out_size, float* dst,
                   int* n_pieces, cudaStream_t stream);

int normalize_u8(const uint8_t* in, int N, int S, float* out, cudaStream_t stream);   // [N,S,S,3] u8 -> [N,3,S,S] f32 in [-1,1]

// ---- retrieval metrics (retrieval_metrics.cu): see include/vited_b200.h vited_retrieval_rows ----
int retrieval_rows(const float* sim, const int* labels, int N, int* n_rel, double* ap_sum, int* top1, int* hits10,
                   int* hits100, cudaStream_t stream);

// ---- solver distance tables (solver_tables.cu): see include/vited_b200.h vited_puzzle_tables ----
int puzzle_tables(const float* scores, int flags, const int* order, int N, uint32_t* asym, long long* min_d,
                  long long* second_d, int* n_cand, int* cand, float* compat, float* mutual, int* best_buddy,
                  cudaStream_t stream);

// ---- training-step kernels (train_ops.cu; SURVEY 8f row 1): see include/vited_b200.h vited_train_* ----
int train_cast_scale(const float* in, act_t* out, size_t n, float scale, cudaStream_t s);
int train_act_axpby(const act_t* x, float* y, size_t n, float alpha, float beta, cudaStream_t s);
int train_f32_axpy(const float* x, float* y, size_t n, float alpha, cudaStream_t s);
int train_transpose(const void* in, int in_is_f32, int ld_in, act_t* out, int ld_out, int R, int C, float scale, cudaStream_t s);
int train_ln_forward(const float* x, const float* w, const float* b, act_t* h, float* stats, int R, int D, float eps, cudaStream_t s);
int train_ln_backward(const float* dh, const float* x, const float* stats, const float* w, float* dx, float* dw, float* db,
                      int R, int D, float alpha, cudaStream_t s);
int train_gelu_forward(const act_t* z, act_t* a, size_t n, cudaStream_t s);
int train_gelu_backward(const float* da, const act_t* z, float* dz, size_t n, cudaStream_t s);
int train_colsum(const float* dy, float* db, int R, int N, float alpha, cudaStream_t s);
int train_gather_rows(const float* in, const int* idx, float* out, int n_blocks, int rows_per, int in_block_stride,
                      int in_row_off, int out_block_stride, int out_row_off, int D, int accumulate, cudaStream_t s);
int train_scatter_add_rows(const float* src, const int* idx, float* dst, int n_blocks, int rows_per, int src_block_stride,
                           int src_row_off, int dst_block_stride, int dst_row_off, int D, float alpha, cudaStream_t s);
// flag non-null (backward only): *flag = 1 when a dS value of the tensor-core kernels does not survive its conversion to
// the 16-bit type (kActRangeLimit); the fp32 SIMT kernels convert nothing and never touch it
int train_attention(int backward, const act_t* q, int q_ld, const act_t* k, int k_ld, const act_t* v, int v_ld, act_t* o,
                    int o_ld, float* lse, const float* d_o, int do_ld, float* dsum, float* dq, int dq_ld, float* dk, int dk_ld,
                    float* dv, int dv_ld, int n_seq, int H, int hd, int Tq, int Tk, float scale, cudaStream_t s,
                    int* flag = nullptr);
// tensor-core (wmma) version of train_attention for head_dim 32 / 64 (train_attn.cu); the backward pass also reads the
// forward output o (D_i = do_i . o_i)
bool train_attention_wmma_supported(int hd);
int train_attention_wmma(int backward, const act_t* q, int q_ld, const act_t* k, int k_ld, const act_t* v, int v_ld, act_t* o,
                         int o_ld, float* lse, const float* d_o, int do_ld, float* dsum, float* dq, int dq_ld, float* dk,
                         int dk_ld, float* dv, int dv_ld, int n_seq, int H, int hd, int Tq, int Tk, float scale, cudaStream_t s,
                         int* flag = nullptr);

// ---- the optimiser side of a training iteration (train_optim.cu): see include/vited_b200.h ----
// |x| from which a value does not survive the conversion to the 16-bit type: fp16 conversions saturate at 65504 (f2act),
// bf16 has the fp32 exponent range and loses only non-finite values
#if VITED_ACT_BF16
constexpr float kActRangeLimit = __builtin_huge_valf();
#else
constexpr float kActRangeLimit = 65504.f;
#endif
float train_range_limit();
int train_range_check(const void* x, int is_f32, int64_t n, float limit, int* flag, cudaStream_t s);
int train_grad_norm(const int64_t* table, int n_tensors, double* partials, int n_partials, float* out, cudaStream_t s);
int train_adamw(const int64_t* table, int n_tensors, int64_t max_numel, double lr, double beta1, double beta2, double eps,
                float clip_coef, double bc1, double bc2, cudaStream_t s);
int train_bce_logits(const float* logits, const float* labels, int n, float* loss, float* dlogits, float grad_scale,
                     cudaStream_t s);

// ---- attention (attention.cu) ----
// Sequences live in the split layout. Logical token s of sequence b: s==0 && has_cls ? cls row : patch row.
struct AttnArgs {
  const act_t* q; int q_ld;      // row stride in elements
  const act_t* k; int k_ld;
  const act_t* v; int v_ld;
  act_t* o; int o_ld;
  int n_seq;                    // number of query sequences (pairs / items)
  int n_heads, head_dim;
  int nq_patch, q_has_cls;      // query tokens per sequence = nq_patch + q_has_cls
  int nk_patch, k_has_cls;      // key tokens per sequence
  int n_kv_seq;                 // number of key/value sequences in the k/v buffers
  const int* kv_index;          // [n_seq] key/value sequence per query sequence; null => identity
  float scale;
};
int attention(const AttnArgs& a, int impl, cudaStream_t stream);
// tcgen05/TMEM kernels for the hot decoder shapes (attention_tc.cu); attention() dispatches to them by itself
bool attention_tc_supported(const AttnArgs& a);
int attention_tc(const AttnArgs& a, cudaStream_t stream);
// puzzle shape with two (sequence, head) units per 128-row tile (attention_pair.cu; -DVITED_EXPERIMENTAL builds only)
bool attention_pair_supported(const AttnArgs& a);
int attention_pair(const AttnArgs& a, cudaStream_t stream);
bool attention_tc_cls_supported(const AttnArgs& a);
int attention_tc_cls(const AttnArgs& a, cudaStream_t stream);
// class-token query only: q and o are the full split-layout buffers (q_has_cls = 1); only their class-token rows
// (row n_seq*nq_patch + b) are read / written. The puzzle-shape warp kernel assumes nq_patch = 64.
int attention_cls(const AttnArgs& a, cudaStream_t stream);

}  // namespace vited
