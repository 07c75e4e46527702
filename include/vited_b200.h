/* vited_b200.h -- C-ABI of the B200-native ViT-ED all-pairs scoring path.
 *
 * The reference (glmanhtu/vit-ed) has no FFI on this path: it sits behind a Python nn.Module API
 *   build_model(config)                                    models/build.py:15-32
 *   VisionTransformerCustom.__init__(img_size, patch_size, in_chans, num_classes, embed_dim, depth, c_depth,
 *                                    num_heads, mlp_ratio, qkv_bias, ...)   models/vision_transformer.py:282-316
 *   VisionTransformerCustom.forward(x, x2=None, forward_first_part=False)   models/vision_transformer.py:412-420
 * and the two pair-grid loops evaluation.py:101-114 and hisfrag.py:189-246 that call it.
 * This header is what a ctypes / cffi binding of a drop-in replacement binds (see INTEGRATION.md); the Python mirror
 * in vit-ed_b200/ keeps the reference's names and argument meaning on top of it.
 *
 * Conventions: all data pointers are DEVICE pointers owned by the caller (torch tensors kept alive by the caller);
 * outputs are caller-allocated; work is enqueued on `stream` (a cudaStream_t passed as void*; NULL = default
 * stream) and is asynchronous with respect to the host unless stated. Every function returns 0 on success and a
 * non-zero status otherwise; vited_last_error() then holds a message. No exceptions cross the boundary. A handle is
 * bound to one device and is not thread-safe (the reference runs one Python thread per GPU process).
 */
#ifndef VITED_B200_H
#define VITED_B200_H

#include <stdint.h>

#if defined(__GNUC__)
#define VITED_API __attribute__((visibility("default")))
#else
#define VITED_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

typedef struct vited_engine vited_engine;

/* Mirrors the constructor arguments build_model() passes (models/build.py:19-32, defaults config.py:68-79). */
typedef struct vited_config {
  int32_t img_size;     /* DATA.IMG_SIZE            */
  int32_t patch_size;   /* MODEL.PJS.PATCH_SIZE     */
  int32_t in_chans;     /* MODEL.PJS.IN_CHANS (3)   */
  int32_t num_classes;  /* MODEL.NUM_CLASSES        */
  int32_t embed_dim;    /* MODEL.PJS.EMBED_DIM      */
  int32_t depth;        /* MODEL.PJS.DEPTH          */
  int32_t c_depth;      /* MODEL.PJS.C_DEPTH        */
  int32_t num_heads;    /* MODEL.PJS.NUM_HEADS      */
  float mlp_ratio;      /* MODEL.PJS.MLP_RATIO      */
  int32_t qkv_bias;     /* MODEL.PJS.QKV_BIAS       */
} vited_config;

/* Grid modes of vited_score_grid. */
enum {
  /* puzzle: ordered pairs (i, j), i != j, i-major -- data/datasets/pieces_dataset.py:27-32 */
  VITED_GRID_ORDERED_OFFDIAG = 0,
  /* Hisfrag: pairs (a, b), a <= b, a-major, diagonal included -- hisfrag.py:166-167 (torch.combinations) */
  VITED_GRID_UPPER_TRI_DIAG = 1
};

/* Options for vited_set_option. */
enum {
  VITED_OPT_GEMM_IMPL = 0,      /* 0 = tcgen05/TMA kernel (default), 1 = SIMT debugging reference kernel        */
  VITED_OPT_ATTN_IMPL = 1,      /* 0 = default (tcgen05/TMEM kernel where the shape has one, else the mma.sync flash
                                   kernel), 1 = SIMT debugging reference kernel, 2 = mma.sync flash kernel always   */
  VITED_OPT_CHUNK_ROWS = 2,     /* target token rows per decoder chunk (default 524288)                          */
  VITED_OPT_CACHE_LAYER0 = 3,   /* 1 (default) = run decoder layer 0's self-attention once per item, not per pair */
  VITED_OPT_PROFILE = 4,        /* 1 = record a CUDA event before every launch (see vited_profile_json); default 0   */
  VITED_OPT_PRUNE_TAIL = 5,     /* 1 (default) = in the last decoder layer run everything after the K/V projection of
                                   its self-attention on the class-token rows only (only row 0 reaches the head)   */
  VITED_OPT_FUSE_LN = 6,        /* 1 (default) = residual add + LayerNorm run in the epilogue of the producing GEMM
                                   (embed_dim 384, large row counts); 0 = separate resid_ln kernel                  */
  VITED_OPT_KV_BUDGET_MB = 7,   /* vited_score_grid processes context rows in blocks whose K/V cache (all decoder
                                   layers) fits this many MB (default 8000; Hisfrag: 18.9 MB per fragment)          */
  VITED_OPT_FUSE_MLP = 8,       /* 1 (default) = the MLP sub-block (fc1, GELU, fc2), its residual add and the next
                                   layer's LayerNorm run in one kernel, hidden activations never written (needs
                                   FUSE_LN; embed_dim 384, large row counts); 0 = fc1 GEMM + fused fc2 GEMM          */
  VITED_OPT_XSRC_BUDGET_MB = 9  /* vited_score_grid(_u8) holds the decoder input states of at most this many MB of grid
                                   columns at once (default 32000; (N_e + 1) * embed_dim * 4 bytes per column item,
                                   Hisfrag: 1.57 MB). When all columns of a call fit, they are built once up front;
                                   otherwise they are rebuilt per window of columns for every K/V row block (at least
                                   one column per window). Same scores either way, up to fp32 rounding noise of the
                                   different chunk shapes.                                                         */
};

/* Library-wide last error message (thread-local). */
VITED_API const char* vited_last_error(void);

/* replaces: VisionTransformerCustom.__init__ (models/vision_transformer.py:282-376) + model.cuda() (evaluation.py:60) */
VITED_API int vited_create(const vited_config* cfg, int device, vited_engine** out);
VITED_API void vited_destroy(vited_engine* e);
VITED_API int vited_set_option(vited_engine* e, int option, int64_t value);

/* replaces: load_pretrained -> model.load_state_dict (misc/utils.py:48-127). `name` is the state_dict key
 * (e.g. "cross_blocks.3.cross_attn.kv.weight"), `data` a device pointer to the fp32 tensor in PyTorch layout
 * (Linear weights [out, in], conv weight [D, C, p, p]); the engine packs its own 16-bit copy, the caller's tensor is
 * only borrowed for the duration of the call (synchronises `stream`). Unknown keys are an error. */
VITED_API int vited_load_weight(vited_engine* e, const char* name, const float* data, int64_t numel, void* stream);
/* number of state_dict tensors the engine expects / has received; forward calls fail until they match */
VITED_API int vited_num_weights_expected(vited_engine* e);
VITED_API int vited_num_weights_loaded(vited_engine* e);
/* i-th expected state_dict key (0 <= i < expected), NULL if out of range */
VITED_API const char* vited_weight_name(vited_engine* e, int i);

/* replaces: model(x, forward_first_part=True) -- forward_first_part, models/vision_transformer.py:382-388
 * images [B, in_chans, S, S] f32 -> tokens [B, N_e, D] f32 (no cls token, no final norm). */
VITED_API int vited_encode(vited_engine* e, const float* images, int B, float* out_tokens, void* stream);

/* replaces: model(x1_tokens, x2_images) -- forward_second_part + forward_head, vision_transformer.py:403-405, :415-417
 * ctx_tokens [B, N_e, D] f32, images [B, in_chans, S, S] f32 -> logits [B, num_classes] f32. */
VITED_API int vited_decode(vited_engine* e, const float* ctx_tokens, const float* images, int B, float* out_logits,
                 void* stream);

/* replaces: model(pairs) one-shot -- forward_features + forward_head, vision_transformer.py:407-410, :418-420
 * pairs [B, 2, in_chans, S, S] f32 -> logits [B, num_classes] f32. */
VITED_API int vited_forward_pairs(vited_engine* e, const float* pairs, int B, float* out_logits, void* stream);

/* replaces: the pair-grid loops evaluation.py:101-114 (mode ORDERED_OFFDIAG) and hisfrag.py:189-231 (mode
 * UPPER_TRI_DIAG), for grid rows [row_begin, row_end) of an N-item grid.
 * images [N, in_chans, S, S] f32 (all items, every rank holds them);
 * out    [row_end - row_begin, N, num_classes] f32, out[(i - row_begin), j, :] = logits of pair (ctx = i, x2 = j).
 * Entries that are not part of the mode's pair set (the diagonal, or j < i) are left untouched. */
VITED_API int vited_score_grid(vited_engine* e, const float* images, int N, int mode, int row_begin, int row_end, float* out,
                     void* stream);
/* vited_score_grid on the decoded bytes: images [N, S, S, in_chans] u8 (HWC, the crops a dataset yields; 1 byte per
 * value against 4 for the f32 form, e.g. 0.79 MB against 3.15 MB per 512 x 512 RGB fragment); ToTensor +
 * Normalize(.5, .5) (hisfrag.py:89-93, data/transforms.py:12-26) is applied while the patch matrix is formed, with the
 * arithmetic of vited_normalize_u8, so the result is bit-identical to vited_score_grid on the normalised f32 images.
 * Built for in_chans 3 and patch sizes 4, 8, 16, 32. Everything else as vited_score_grid.
 * Device memory of one call beyond the images: the decoder input states of the columns, (N_e + 1) * embed_dim * 4
 * bytes per column item, at most VITED_OPT_XSRC_BUDGET_MB; the K/V cache of one row block, at most
 * VITED_OPT_KV_BUDGET_MB; and a workspace of about one decoder chunk (VITED_OPT_CHUNK_ROWS token rows). */
VITED_API int vited_score_grid_u8(vited_engine* e, const uint8_t* images, int N, int mode, int row_begin, int row_end,
                                  float* out, void* stream);

/* replaces: the `sub_pairs` batches of hisfrag.py:221-229 and a one-shot pass over a pair dataset -- any pair list, with
 * every item encoded and its decoder input state built once per call, as the grid does.
 * images [N, in_chans, S, S] f32 (vited_score_pairs) or [N, S, S, in_chans] u8 (vited_score_pairs_u8, the format and
 * normalisation of vited_score_grid_u8);
 * pairs  [n_pairs, 2] i32 (device): (context item a, decoder item b), indices into images[0..N);
 * out    [n_pairs, num_classes] f32: out[p] = logits of model(tokens(images[a]), images[b]), the (a, b) entry of
 *        vited_score_grid. Any order; duplicates, a == b and a > b are allowed.
 * Only the items the list references are read and computed: its distinct context items in blocks of at most
 * VITED_OPT_KV_BUDGET_MB of K/V cache, its distinct decoder items in windows of at most VITED_OPT_XSRC_BUDGET_MB of
 * decoder input states. Pairs are bucketed by (block, window) on the device with a stable sort, so the same list always
 * gives the same bits; a dense grid's own pair set in its i-major order gives vited_score_grid's bits.
 * Synchronises `stream` once (to size its loops); an index outside [0, N) is an error reported before anything is
 * scored (out untouched), its message names the first such pair. n_pairs == 0 does nothing; n_pairs > INT32_MAX is an
 * error. Device memory of one call: about 20 bytes per pair (the caller's list and three sorted index arrays), 24 bytes
 * per item of N, on top of what vited_score_grid holds. */
VITED_API int vited_score_pairs(vited_engine* e, const float* images, int N, const int32_t* pairs, int64_t n_pairs,
                                float* out, void* stream);
VITED_API int vited_score_pairs_u8(vited_engine* e, const uint8_t* images, int N, const int32_t* pairs,
                                   int64_t n_pairs, float* out, void* stream);

/* number of kernels launched by this engine since creation (bench.py's gpu_launches) */
VITED_API int64_t vited_launch_count(vited_engine* e);
/* Per-kernel-class device time since profiling was switched on / last read, as a JSON object
 * {"<class>": {"ms":, "flops":, "bytes":, "launches":}, ...} (algorithmic flops / bytes of the launches). Synchronises
 * `stream`, resets the counters. The string is owned by the engine and valid until the next call. */
VITED_API const char* vited_profile_json(vited_engine* e, void* stream);
/* 16-bit type of the GEMM / attention operands and of the buffers of the single-kernel entry points below:
 * 0 = IEEE fp16 (default; the reference's autocast dtype, config.py:216), 1 = bf16 (-DVITED_ACT_BF16=1 builds).
 * Accumulators, the residual stream, LayerNorm statistics and softmax are fp32 in both. */
VITED_API int vited_act_dtype(void);
/* bytes of device workspace currently held */
VITED_API int64_t vited_workspace_bytes(vited_engine* e);

/* ---- producer side of the puzzle grid (SURVEY 8f row 2) ----
 * replaces: the per-piece preparation PiecesDataset.__getitem__ + TwoImgSyncEval run 2*N*(N-1) times in DataLoader
 * workers (data/datasets/pieces_dataset.py:34-56, data/transforms.py:12-26): cv2.cvtColor(LAB2RGB) on the eroded
 * piece, PIL bilinear Resize(out_size), ToTensor, Normalize(.5, .5) -- and the crop of Puzzle.make_pieces
 * (paikin_tal_solver/puzzle_importer.py:196-232, :430-446). Once per piece, on the device, bit-identical floats.
 * lab_image [H, W, 3] u8 (device): the puzzle image after cv2.COLOR_BGR2LAB (puzzle_importer.py:136-156);
 * piece_width: grid = floor(H / w) x floor(W / w), centred; side / off: eroded piece side and crop offset
 * (ceil(w * (1 - erosion)) and Python round((w - side) / 2): computed by the caller, vit-ed_b200/pieces.py);
 * out [rows * cols, 3, out_size, out_size] f32 in piece-id (row-major) order; *n_pieces (host, may be NULL) = rows * cols. */
VITED_API int vited_prepare_pieces(const uint8_t* lab_image, int H, int W, int piece_width, int side, int off, int out_size,
                                   float* out, int* n_pieces, void* stream);

/* replaces: ToTensor + Normalize(.5, .5) of the Hisfrag test transform (hisfrag.py:89-93, applied by
 * HisFrag20Test.__getitem__, hisfrag_dataset.py:181-191) after its CenterCrop, which the caller does on the bytes.
 * images [N, S, S, 3] u8 (device) -> out [N, 3, S, S] f32 = (v / 255 - 0.5) / 0.5, bit-identical to torch's fp32 ops. */
VITED_API int vited_normalize_u8(const uint8_t* images, int N, int S, float* out, void* stream);

/* ---- Hisfrag training step (SURVEY 8f row 1) ----
 * replaces: the compute of HisfragTrainer.train_step (hisfrag.py:149-159: encode the batch, decode the pairs
 * model(tokens[groups[:, 1]], samples[groups[:, 0]]), nn.BCEWithLogitsLoss :60-61) and of the backward pass that
 * misc/engine.py:189-257 runs through autograd. The host side (vit-ed_b200/train.py) walks the layers and calls these
 * single-kernel entry points; every Linear (forward, dgrad dX = dY W, wgrad dW = dY^T X) is vited_op_gemm on the tcgen05
 * kernel with 16-bit operands (h16), fed by the transposes below; everything elementwise is fp32. Plain row-major
 * [rows, cols] buffers, sequences as consecutive token rows with the class token first. All pointers are device
 * pointers; `alpha` arguments fold the loss-scale removal into the accumulation of parameter gradients.
 *   cast:        out h16 = in f32 * scale                      axpby16: y f32 = alpha * x h16 + beta * y
 *   axpy32:      y += alpha * x (f32)                          transpose: out h16 [C, ld_out] = scale * in[R, C]^T (f32 or
 *                                                              h16 input), rows R..ld_out-1 of the K dimension zero filled
 *   ln_forward:  h h16 = LayerNorm(x f32) * w + b, stats[r] = (mean, rstd)
 *   ln_backward: dx += d LN / dx (dh f32); dw += alpha * sum dh * xhat; db += alpha * sum dh
 *   gelu_forward / gelu_backward: exact-erf GELU on h16 z; dz f32 = da f32 * gelu'(z)
 *   colsum:      db[c] += alpha * sum_r dy[r, c]
 *   gather_rows / scatter_add_rows: blocks of rows_per consecutive rows moved between [block idx[b]] of one buffer and
 *                block b of the other (pairs <-> items; position / class-token broadcast and its gradient)
 *   attention:   softmax(q k^T * scale) v per (sequence, head) on the warp-level tensor cores (wmma, fp32 accumulation;
 *                head_dim 32 / 64), flash style: the forward stores o h16 and lse [n_seq, H, Tq] (log-sum-exp per query
 *                row); backward = 1 takes o, lse and d_o f32, recomputes the probabilities block by block (nothing
 *                quadratic is stored, no atomics), writes dsum [n_seq, H, Tq] = do . o and accumulates dq, dk, dv (+=, f32)
 *   bce_logits:  loss = mean BCE-with-logits; dlogits = (sigmoid(logit) - label) * grad_scale / n */
VITED_API int vited_train_cast(const float* in, void* out, int64_t n, float scale, void* stream);
VITED_API int vited_train_axpby16(const void* x, float* y, int64_t n, float alpha, float beta, void* stream);
VITED_API int vited_train_axpy32(const float* x, float* y, int64_t n, float alpha, void* stream);
VITED_API int vited_train_transpose(const void* in, int in_is_f32, int ld_in, void* out, int ld_out, int R, int C,
                                    float scale, void* stream);
VITED_API int vited_train_ln_forward(const float* x, const float* w, const float* b, void* h, float* stats, int R, int D,
                                     float eps, void* stream);
VITED_API int vited_train_ln_backward(const float* dh, const float* x, const float* stats, const float* w, float* dx,
                                      float* dw, float* db, int R, int D, float alpha, void* stream);
VITED_API int vited_train_gelu_forward(const void* z, void* a, int64_t n, void* stream);
VITED_API int vited_train_gelu_backward(const float* da, const void* z, float* dz, int64_t n, void* stream);
VITED_API int vited_train_colsum(const float* dy, float* db, int R, int N, float alpha, void* stream);
VITED_API int vited_train_gather_rows(const float* in, const int32_t* idx, float* out, int n_blocks, int rows_per,
                                      int in_block_stride, int in_row_off, int out_block_stride, int out_row_off, int D,
                                      int accumulate, void* stream);
VITED_API int vited_train_scatter_add_rows(const float* src, const int32_t* idx, float* dst, int n_blocks, int rows_per,
                                           int src_block_stride, int src_row_off, int dst_block_stride, int dst_row_off,
                                           int D, float alpha, void* stream);
VITED_API int vited_train_attention(int backward, const void* q, int q_ld, const void* k, int k_ld, const void* v, int v_ld,
                                    void* o, int o_ld, float* lse, const float* d_o, int do_ld, float* dsum, float* dq,
                                    int dq_ld, float* dk, int dk_ld, float* dv, int dv_ld, int n_seq, int H, int hd, int Tq,
                                    int Tk, float scale, void* stream);
VITED_API int vited_train_bce_logits(const float* logits, const float* labels, int n, float* loss, float* dlogits,
                                     float grad_scale, void* stream);

/* ---- Hisfrag training iteration: overflow detection, gradient clipping, AdamW ----
 * The 16-bit conversions of this library saturate (fp16 at +-65504) instead of producing inf, so an overflowing
 * loss-scaled gradient is finite and silently wrong; these entry points let the host detect it, skip the step and back
 * off the scale (vit-ed_b200/train.py train_iteration). `flag` is one int32 on the device, sticky: entry points set it
 * to 1 and never clear it.
 *   range_limit: |x| from which a value does not survive the 16-bit conversion: 65504 (fp16 builds) or +inf (bf16
 *                builds, where only non-finite values count)
 *   range_check: *flag = 1 if any of x[0, n) (f32 if is_f32, else h16) is non-finite or has |x| >= limit; any element
 *                offset and any n >= 0
 *   attention_chk: vited_train_attention, and in the backward pass *flag = 1 when a dS = P (dP - D) scale value of the
 *                tensor-core kernels is out of range before its conversion to h16 (|dS| can reach about
 *                2 |dO_i| max_j |V_j| scale with dO in range). flag NULL = vited_train_attention. The fp32 kernels of
 *                other head dims convert nothing and leave the flag alone. */
/* replaces: the found_inf check of GradScaler (torch.amp, misc/engine.py:189-257) */
VITED_API float vited_train_range_limit(void);
VITED_API int vited_train_range_check(const void* x, int is_f32, int64_t n, float limit, int32_t* flag, void* stream);
/* replaces: the backward of the attention (misc/engine.py:189-257 autograd) with GradScaler's overflow check */
VITED_API int vited_train_attention_chk(int backward, const void* q, int q_ld, const void* k, int k_ld, const void* v,
                                        int v_ld, void* o, int o_ld, float* lse, const float* d_o, int do_ld, float* dsum,
                                        float* dq, int dq_ld, float* dk, int dk_ld, float* dv, int dv_ld, int n_seq, int H,
                                        int hd, int Tq, int Tk, float scale, int32_t* flag, void* stream);
/* replaces: the total norm of clip_grad_norm_(params, 5.0) (misc/utils.py:206-226).
 * table [n_tensors, 2] int64 on the device: (pointer to f32 gradient, numel) per tensor. Sum of squares in fp64 over a
 * fixed partition (n_partials blocks, partials [n_partials] f64 workspace) and a fixed-order final sum: bit-reproducible
 * for a given table and n_partials. out_sumsq_and_flag: 8 bytes, 8-byte aligned: out[0] = (float) sum of squares, the
 * int32 after it is a sticky flag set to 1 when that value is non-finite. */
VITED_API int vited_train_grad_norm(const int64_t* table, int n_tensors, double* partials, int n_partials,
                                    float* out_sumsq_and_flag, void* stream);
/* replaces: optimizer.step() of torch.optim.AdamW (misc/optimizer.py:12-46) after clip_grad_norm_.
 * table [n_tensors, 6] int64 on the device: (param, grad, exp_avg, exp_avg_sq pointers (f32, numel elements each),
 * numel, weight decay as the bit pattern of a double) per tensor; max_numel = the largest numel. One step of the
 * single-tensor form of torch.optim.AdamW operation for operation, with g = grad * clip_coef:
 *   p *= 1 - lr wd;  m = lerp(m, g, 1 - beta1);  v = beta2 v + (1 - beta2) g^2;
 *   p -= (lr / bias_correction1) m / (sqrt(v) / sqrt(bias_correction2) + eps)
 * with bias_correction{1,2} = 1 - beta{1,2}^t computed by the caller in double. grad is read, never written. */
VITED_API int vited_train_adamw(const int64_t* table, int n_tensors, int64_t max_numel, double lr, double beta1,
                                double beta2, double eps, float clip_coef, double bias_correction1,
                                double bias_correction2, void* stream);

/* ---- consumer side of the puzzle grid (SURVEY 8f row 3) ----
 * replaces: the tables InterPieceDistance.__init__ fills through 4*N*(N-1) callbacks into evaluation.py:116-131's
 * distance_function -- PieceDistanceInformation.calculate_inter_piece_distances (paikin_tal_solver/
 * inter_piece_distance.py:189-240: uint32 distances, minimum / second best, best-buddy candidates),
 * calculate_asymmetric_compatibility (:325-372), InterPieceDistance.calculate_mutual_compatibility (:489-524) and the
 * candidate matching of find_best_buddies (:626-648), for a type-1 puzzle (neighbour side = complementary side).
 * scores  [N, N, 4] f32 indexed by origin piece id;
 * flags   bit 0 (VITED_TABLES_LOGITS): scores are logits and 1 - sigmoid is applied as evaluation.py:109-114 does
 *         (clear: scores already are the distances 1 - sigmoid(logit));
 *         bit 1 (VITED_TABLES_F32_PRODUCT): `pred[k] * 1000.` (evaluation.py:118-129, np.float32 scalar x Python float)
 *         is evaluated in float32 as NumPy >= 2 does. Clear (default): in float64, as the NumPy 1.x of the reference's
 *         pinned stack (requirements.txt: torch~=2.1, scipy~=1.9.1) does -- the truncated uint32 distance differs by one
 *         on ~1e-5 of the entries between the two;
 * order   [N] i32 origin id of the piece at list position k (evaluation.py:87 shuffles the list), NULL = identity;
 * All outputs are indexed by list position, rows (i, side) with side = PuzzlePieceSide value (top 0, right 1,
 * bottom 2, left 3):  asym_dist [N,4,N] u32 (diagonal 2^31-1), min_dist / second_dist [N,4] i64 (sys.maxsize - 1 /
 * sys.maxsize where the reference leaves its initial values), n_candidates [N,4] i32 = pieces at the minimum,
 * candidate [N,4] i32 = the lowest such j (-1 if none), asym_compat / mutual_compat [N,4,N] f32 (diagonal +inf),
 * best_buddy [N,4] i32 = j or -1. Every value is bit-identical to the reference's under the selected scalar rules. */
#define VITED_TABLES_LOGITS 1
#define VITED_TABLES_F32_PRODUCT 2
VITED_API int vited_puzzle_tables(const float* scores, int flags, const int32_t* order, int N,
                                  uint32_t* asym_dist, int64_t* min_dist, int64_t* second_dist, int32_t* n_candidates,
                                  int32_t* candidate, float* asym_compat, float* mutual_compat, int32_t* best_buddy,
                                  void* stream);

/* ---- consumer side of the fragment grid (SURVEY 8f row 4) ----
 * replaces: wi19_evaluate.get_metrics(distance_matrix, labels) (misc/wi19_evaluate.py:12-56) as hisfrag.py:306-309 calls
 * it on distance = 1 - fp16(similarity) (hisfrag.py:283-296): per query row i, with the first sorted column dropped
 * (:29-30) and relevance = same label (:26-27, self included),
 *   n_relevant[i]  relevant items left,           ap_sum[i]  sum of precision-at-rank over them (f64),
 *   top1[i]        1 if the nearest remaining item is relevant,   hits10 / hits100[i]  relevant items within rank 10 / 100.
 * mAP = mean over rows with n_relevant > 0 of ap_sum / n_relevant; top-1 = mean(top1); Pr@k = mean(hits_k /
 * min(n_relevant, k)) (0 / 0 = nan for singleton queries, as in the reference). Equal distances are ordered by
 * ascending index (numpy's argsort leaves the order of ties to its implementation).
 * sim [N, N] f32 (device): the logits of vited_score_grid mode UPPER_TRI_DIAG after mirroring; labels [N] i32. */
VITED_API int vited_retrieval_rows(const float* sim, const int32_t* labels, int N, int32_t* n_relevant, double* ap_sum,
                                   int32_t* top1, int32_t* hits10, int32_t* hits100, void* stream);

/* ---- single-kernel entry points (used by tests/ and profiles/ to check and time each kernel in isolation) ---- */
/* ("h16" = the 16-bit type vited_act_dtype() names) C[M,N] h16 = act(A[M,K] h16 * W[N,K]^T h16 + bias[N] f32); act: 0 none, 1 exact-erf GELU; impl as GEMM_IMPL */
VITED_API int vited_op_gemm(const void* A, const void* W, const float* bias, void* C, int M, int N, int K, int act, int impl,
                  void* stream);
/* fused Linear + residual + LayerNorm (N must be 384): x[M,384] f32 += A[M,K] h16 * W[384,K]^T h16 + bias;
 * h[M,384] h16 = LayerNorm(x) * ln_w + ln_b */
VITED_API int vited_op_gemm_resid_ln(const void* A, const void* W, const float* bias, float* x, const float* ln_w,
                           const float* ln_b, void* h, int M, int N, int K, float eps, void* stream);
/* fused MLP sub-block + residual + LayerNorm (D must be 384, hidden a multiple of 64): x[M,384] f32 +=
 * GELU(h_in[M,384] h16 * W1[hidden,384]^T + b1) * W2[384,hidden]^T + b2; h_out[M,384] h16 = LayerNorm(x) * ln_w + ln_b
 * (timm Mlp inside Block / CrossBlock, vision_transformer.py:126, :272, + the next norm1). h_out may alias h_in. */
VITED_API int vited_op_mlp_resid_ln(const void* h_in, const void* W1, const float* b1, const void* W2, const float* b2,
                          float* x, const float* ln_w, const float* ln_b, void* h_out, int M, int D, int hidden,
                          float eps, void* stream);
/* the cross-attention projection + residual + norm2 in front of the fused MLP sub-block (D must be 384, hidden a
 * multiple of 64): x_mid = x + o[M,384] h16 * Wp[384,384]^T h16 + bp; h = LayerNorm(x_mid) * ln2_w + ln2_b (h16);
 * x[M,384] f32 = x_mid + GELU(h * W1^T + b1) * W2^T + b2; h_out[M,384] h16 = LayerNorm(x) * ln_w + ln_b
 * (a decoder CrossBlock's cross_attn.proj and Mlp, vision_transformer.py:271-272, + the next norm1). x_mid and h are
 * never written: on return x holds the block's output rows. */
VITED_API int vited_op_cproj_mlp_resid_ln(const void* o, const void* Wp, const float* bp, float* x, const float* ln2_w,
                                const float* ln2_b, const void* W1, const float* b1, const void* W2, const float* b2,
                                const float* ln_w, const float* ln_b, void* h_out, int M, int D, int hidden, float eps,
                                void* stream);
/* x += delta (h16, may be NULL); h = LayerNorm(x) * w + b as h16 (w NULL => skipped). Split token layout. */
VITED_API int vited_op_resid_ln(float* x, const void* delta, const float* ln_w, const float* ln_b, void* h, int n_seq,
                      int n_patch, int has_cls, int D, float eps, void* stream);
/* q/k/v/o h16 in the split token layout; kv_index NULL => identity */
VITED_API int vited_op_attention(const void* q, int q_ld, const void* k, int k_ld, const void* v, int v_ld, void* o, int o_ld,
                       int n_seq, int n_heads, int head_dim, int nq_patch, int q_has_cls, int nk_patch,
                       int k_has_cls, int n_kv_seq, const int32_t* kv_index, float scale, int impl, void* stream);
/* class-token query only (the pruned last decoder layer, vision_transformer.py:397-401: only token 0 reaches the head).
 * q and o are full split-layout buffers of n_seq sequences of nk_patch patch rows + a class token; only their class-token
 * rows (row n_seq*nk_patch + b) are read and written. k / v as in vited_op_attention. */
VITED_API int vited_op_attention_cls(const void* q, int q_ld, const void* k, int k_ld, const void* v, int v_ld, void* o,
                                     int o_ld, int n_seq, int n_heads, int head_dim, int nk_patch, int k_has_cls,
                                     int n_kv_seq, const int32_t* kv_index, float scale, void* stream);
/* final LayerNorm + head (vision_transformer.py:400, :417): y = LayerNorm(x[p] + delta[p]) * ln_w + ln_b;
 * out[p*C + c] = y . head_w[c] + head_b[c]. x [P,D] f32, delta [P,D] h16 or NULL, head_w [C,D] f32, all in fp32 math. */
VITED_API int vited_op_head(const float* x, const void* delta, const float* ln_w, const float* ln_b, const float* head_w,
                            const float* head_b, float* out, int P, int D, int C, float eps, void* stream);
/* images [B,C,S,S] f32 -> [B*(S/p)^2, C*p*p] h16 */
VITED_API int vited_op_im2col(const float* images, void* out, int B, int C, int S, int p, void* stream);
/* images [B,S,S,C] u8 -> the same [B*(S/p)^2, C*p*p] h16, bit-identical to vited_normalize_u8 + vited_op_im2col
 * (C = 3, p in {4, 8, 16, 32}; `images` aligned to the largest power of two <= 16 that divides p*C) */
VITED_API int vited_op_im2col_u8(const uint8_t* images, void* out, int B, int C, int S, int p, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* VITED_B200_H */
