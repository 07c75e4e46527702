// Host-side engine behind the C-ABI (include/vited_b200.h): weight packing, workspace, and the launch sequences for
// encode / decode / one-shot / all-pairs grid scoring. Everything here is plumbing around the kernels in
// gemm_tc.cu, attention.cu and rowops.cu; there is no CPU compute path.
//
// Data layout in HBM (see DESIGN.md):
//   * token rows use the "split" layout: n_seq*N_e patch rows followed by n_seq class-token rows, so that 64/1024
//     patch tokens per sequence tile exactly into 64-row attention tiles and GEMMs run over one flat row space;
//   * residual stream x is fp32 [rows, D]; every GEMM operand/result is fp16; sub-block outputs are written as a
//     fp16 `delta` and folded into x by the fused residual+LayerNorm kernel;
//   * per grid: Xsrc = decoder input of every item (after layer-0 self-attention when cached), fp32 split layout;
//     KV[l] = kv(norm_context(enc_tokens)) for the current block of context rows, fp16 [rows*N_e, 2D].
#include "../../include/vited_b200.h"
#include "kernels.h"

#include <cstdarg>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <vector>

namespace vited {

static thread_local char g_err[1024] = "";
void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
const char* get_error() { return g_err; }

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  int ensure(size_t bytes, bool headroom = true) {
    if (bytes <= cap) return 0;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    size_t want = headroom ? bytes + (bytes >> 3) : bytes;  // 12.5% headroom against re-allocation churn
    cudaError_t e = cudaMalloc(&p, want);
    if (e != cudaSuccess) {
      set_error("cudaMalloc(%zu bytes) failed: %s", want, cudaGetErrorString(e));
      return 1;
    }
    cap = want;
    return 0;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
  template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

struct Linear { act_t* w = nullptr; float* b = nullptr; int out = 0, in = 0; };
struct LNorm { float* w = nullptr; float* b = nullptr; };
struct EncBlock { LNorm norm1, norm2; Linear qkv, proj, fc1, fc2; };
struct DecBlock { LNorm norm1, norm_cross, norm_context, norm2; Linear qkv, proj, q, kv, cproj, fc1, fc2; };

struct Slot {
  void* dst;
  bool to_act;
  int64_t numel;
  bool loaded;
};

}  // namespace vited

using namespace vited;

struct vited_engine {
  vited_config cfg;
  int device = 0;
  int D = 0, H = 0, hd = 0, G = 0, Ne = 0, Nd = 0, Kpe = 0, hidden = 0, C = 0;
  float scale = 1.f;
  Linear patch;
  float* pos = nullptr;
  float* cls = nullptr;
  std::vector<EncBlock> enc;
  std::vector<DecBlock> dec;
  LNorm norm;
  float* head_w = nullptr;
  float* head_b = nullptr;
  std::vector<void*> owned;  // weight allocations
  std::map<std::string, Slot> slots;
  std::vector<std::string> names;
  int loaded = 0;
  // options
  int gemm_impl = IMPL_FAST, attn_impl = IMPL_FAST;
  int64_t chunk_rows = 524288;   // measured: 262144 -> 524288 rows per chunk +4.7 % (fewer launch tails), no gain beyond
  int cache_layer0 = 1;
  int prune_tail = 1;   // last decoder layer: only the class-token row continues past self-attention
  int fuse_ln = 1;      // residual + LayerNorm in the epilogue of the N = 384 GEMMs (gemm_ln.cu)
  int fuse_mlp = 1;     // fc1 + GELU + fc2 + residual + LayerNorm in one kernel (mlp_ln.cu); needs fuse_ln
  int kv_budget_mb = 8000;  // K/V cache budget of one block of context rows in vited_score_grid
  int64_t xsrc_budget_mb = 32000;  // decoder input states of one window of grid columns in vited_score_grid
  int64_t launches = 0;
  // optional per-kernel timing (bench.py's roofline): one event before every launch, intervals summed per class
  int profile = 0;
  std::vector<cudaEvent_t> ev_pool;
  size_t ev_used = 0;
  struct ProfRec { cudaEvent_t ev; int cls; double flops; double bytes; };
  std::vector<ProfRec> recs;
  std::vector<std::string> cls_names;
  std::string profile_json;
  // workspace
  DevBuf x, h, qkv, o, q, delta, hid, col, tok, xsrc, enc_tok, kv, ci, xj, tmp_tok;
  DevBuf out_pos, pl_items, pl_hist, pl_info;   // vited_score_pairs: sorted output positions, item maps, sort, info

  int64_t workspace_bytes() const {
    return (int64_t)(x.cap + h.cap + qkv.cap + o.cap + q.cap + delta.cap + hid.cap + col.cap + tok.cap + xsrc.cap +
                     enc_tok.cap + kv.cap + ci.cap + xj.cap + tmp_tok.cap + out_pos.cap + pl_items.cap + pl_hist.cap +
                     pl_info.cap);
  }
};

namespace vited {

#define TRY(expr)            \
  do {                       \
    if ((expr) != 0) return 1; \
  } while (0)

static int alloc_f32(vited_engine* e, float** p, size_t n) {
  VITED_CUDA_OK(cudaMalloc(p, n * sizeof(float)));
  VITED_CUDA_OK(cudaMemset(*p, 0, n * sizeof(float)));
  e->owned.push_back(*p);
  return 0;
}
static int alloc_act(vited_engine* e, act_t** p, size_t n) {
  VITED_CUDA_OK(cudaMalloc(p, n * sizeof(act_t)));
  VITED_CUDA_OK(cudaMemset(*p, 0, n * sizeof(act_t)));
  e->owned.push_back(*p);
  return 0;
}
static void reg(vited_engine* e, const std::string& name, void* dst, bool to_act, int64_t numel) {
  e->slots[name] = Slot{dst, to_act, numel, false};
  e->names.push_back(name);
}
static int make_linear(vited_engine* e, const std::string& prefix, Linear* l, int out, int in, bool bias) {
  l->out = out;
  l->in = in;
  TRY(alloc_act(e, &l->w, (size_t)out * in));
  TRY(alloc_f32(e, &l->b, out));  // stays zero when the reference layer has no bias (qkv_bias=False)
  reg(e, prefix + ".weight", l->w, true, (int64_t)out * in);
  if (bias) reg(e, prefix + ".bias", l->b, false, out);
  return 0;
}
static int make_ln(vited_engine* e, const std::string& prefix, LNorm* n, int D) {
  TRY(alloc_f32(e, &n->w, D));
  TRY(alloc_f32(e, &n->b, D));
  reg(e, prefix + ".weight", n->w, false, D);
  reg(e, prefix + ".bias", n->b, false, D);
  return 0;
}

static int build(vited_engine* e) {
  const vited_config& c = e->cfg;
  VITED_CHECK(c.img_size > 0 && c.patch_size > 0 && c.img_size % c.patch_size == 0,
              "img_size %d must be a positive multiple of patch_size %d", c.img_size, c.patch_size);
  VITED_CHECK(c.embed_dim > 0 && c.num_heads > 0 && c.embed_dim % c.num_heads == 0,
              "dim should be divisible by num_heads (embed_dim=%d num_heads=%d)", c.embed_dim, c.num_heads);
  VITED_CHECK(c.embed_dim % 8 == 0, "embed_dim %d must be a multiple of 8", c.embed_dim);
  VITED_CHECK(c.depth >= 1 && c.c_depth >= 1 && c.num_classes >= 1 && c.in_chans >= 1, "bad depth/classes/channels");
  e->D = c.embed_dim;
  e->H = c.num_heads;
  e->hd = e->D / e->H;
  VITED_CHECK(e->hd == 32 || e->hd == 64, "head_dim %d unsupported (the attention kernels are built for 32 and 64)",
              e->hd);
  e->G = c.img_size / c.patch_size;
  e->Ne = e->G * e->G;
  e->Nd = e->Ne + 1;
  e->Kpe = c.in_chans * c.patch_size * c.patch_size;
  e->hidden = (int)(c.embed_dim * c.mlp_ratio);
  VITED_CHECK(e->hidden % 8 == 0 && e->Kpe % 8 == 0, "hidden %d / patch K %d must be multiples of 8", e->hidden, e->Kpe);
  e->C = c.num_classes;
  e->scale = 1.0f / sqrtf((float)e->hd);
  const int D = e->D;
  const bool qb = c.qkv_bias != 0;

  TRY(alloc_f32(e, &e->cls, D));
  reg(e, "cls_token", e->cls, false, D);
  TRY(alloc_f32(e, &e->pos, (size_t)e->Nd * D));
  reg(e, "pos_embed", e->pos, false, (int64_t)e->Nd * D);
  TRY(make_linear(e, "patch_embed.proj", &e->patch, D, e->Kpe, true));
  e->enc.resize(c.depth);
  for (int l = 0; l < c.depth; ++l) {
    const std::string p = "blocks." + std::to_string(l);
    EncBlock& b = e->enc[l];
    TRY(make_ln(e, p + ".norm1", &b.norm1, D));
    TRY(make_linear(e, p + ".attn.qkv", &b.qkv, 3 * D, D, qb));
    TRY(make_linear(e, p + ".attn.proj", &b.proj, D, D, true));
    TRY(make_ln(e, p + ".norm2", &b.norm2, D));
    TRY(make_linear(e, p + ".mlp.fc1", &b.fc1, e->hidden, D, true));
    TRY(make_linear(e, p + ".mlp.fc2", &b.fc2, D, e->hidden, true));
  }
  e->dec.resize(c.c_depth);
  for (int l = 0; l < c.c_depth; ++l) {
    const std::string p = "cross_blocks." + std::to_string(l);
    DecBlock& b = e->dec[l];
    TRY(make_ln(e, p + ".norm1", &b.norm1, D));
    TRY(make_linear(e, p + ".attn.qkv", &b.qkv, 3 * D, D, qb));
    TRY(make_linear(e, p + ".attn.proj", &b.proj, D, D, true));
    TRY(make_ln(e, p + ".norm_cross", &b.norm_cross, D));
    TRY(make_ln(e, p + ".norm_context", &b.norm_context, D));
    TRY(make_linear(e, p + ".cross_attn.q", &b.q, D, D, qb));
    TRY(make_linear(e, p + ".cross_attn.kv", &b.kv, 2 * D, D, qb));
    TRY(make_linear(e, p + ".cross_attn.proj", &b.cproj, D, D, true));
    TRY(make_ln(e, p + ".norm2", &b.norm2, D));
    TRY(make_linear(e, p + ".mlp.fc1", &b.fc1, e->hidden, D, true));
    TRY(make_linear(e, p + ".mlp.fc2", &b.fc2, D, e->hidden, true));
  }
  TRY(make_ln(e, "norm", &e->norm, D));
  TRY(alloc_f32(e, &e->head_w, (size_t)e->C * D));
  TRY(alloc_f32(e, &e->head_b, e->C));
  reg(e, "head.weight", e->head_w, false, (int64_t)e->C * D);
  reg(e, "head.bias", e->head_b, false, e->C);
  return 0;
}

// ------------------------------------------------------------------------------------------------------------
// launch helpers (count every kernel for bench.py's gpu_launches)
// ------------------------------------------------------------------------------------------------------------
static int prof_class(vited_engine* e, const std::string& name) {
  for (size_t i = 0; i < e->cls_names.size(); ++i)
    if (e->cls_names[i] == name) return (int)i;
  e->cls_names.push_back(name);
  return (int)e->cls_names.size() - 1;
}
static void prof_mark(vited_engine* e, const char* name, double flops, double bytes, cudaStream_t s) {
  e->launches++;
  if (!e->profile) return;
  if (e->ev_used == e->ev_pool.size()) {
    cudaEvent_t ev;
    cudaEventCreate(&ev);
    e->ev_pool.push_back(ev);
  }
  cudaEvent_t ev = e->ev_pool[e->ev_used++];
  cudaEventRecord(ev, s);
  e->recs.push_back({ev, prof_class(e, name), flops, bytes});
}

static int L_gemm(vited_engine* e, const act_t* A, const Linear& l, act_t* Cout, int M, int act, cudaStream_t s) {
  if (e->profile) {
    char nm[64];
    snprintf(nm, sizeof(nm), "gemm_n%d_k%d%s", l.out, l.in, act == ACT_GELU ? "_gelu" : "");
    prof_mark(e, nm, 2.0 * M * (double)l.out * l.in, 2.0 * ((double)M * l.in + (double)l.out * l.in + (double)M * l.out), s);
  } else {
    e->launches++;
  }
  return gemm_act(A, l.w, l.b, Cout, M, l.out, l.in, act, e->gemm_impl, s);
}
// fused x += A W^T + b; h = LN(x)  (gemm_ln.cu). Caller has checked use_fused_ln().
static bool use_fused_ln(vited_engine* e, size_t rows, const Linear& l) {
  return e->fuse_ln && e->gemm_impl == IMPL_FAST && rows >= 8192 && gemm_resid_ln_supported((int)rows, l.out, l.in);
}
static int L_gemm_ln(vited_engine* e, const act_t* A, const Linear& l, float* x, const LNorm& ln, act_t* h, int M,
                     cudaStream_t s) {
  if (e->profile) {
    char nm[64];
    snprintf(nm, sizeof(nm), "gemm_ln_n%d_k%d", l.out, l.in);
    prof_mark(e, nm, 2.0 * M * (double)l.out * l.in,
              2.0 * ((double)M * l.in + (double)l.out * l.in) + (double)M * l.out * (4.0 + 4.0 + 2.0), s);
  } else {
    e->launches++;
  }
  return gemm_resid_ln(A, l.w, l.b, x, ln.w, ln.b, h, M, l.out, l.in, 1e-6f, s);
}
// fused x += cproj(o); x += fc2(GELU(fc1(norm2(x)))) ; h = LN(x)  (mlp_ln.cu)
static bool use_fused_mlp(vited_engine* e, size_t rows, const Linear& cproj, const Linear& fc1, const Linear& fc2) {
  return e->fuse_mlp && use_fused_ln(e, rows, fc2) && use_fused_ln(e, rows, cproj) && cproj.out == e->D &&
         fc1.in == e->D && fc2.in == fc1.out && cproj_mlp_resid_ln_supported((int)rows, e->D, cproj.in, fc1.out);
}
static int L_cproj_mlp_ln(vited_engine* e, const act_t* o, const Linear& cproj, const LNorm& norm2, const Linear& fc1,
                          const Linear& fc2, float* x, const LNorm& ln, act_t* h_out, int M, cudaStream_t s) {
  if (e->profile) {
    // the name starts with mlp_ln: bench.py's mlp_ln family. Bytes: o (2) + x (4) in, x (4) + h (2) out per element
    char nm[64];
    snprintf(nm, sizeof(nm), "mlp_ln_cproj_d%d_h%d", fc1.in, fc1.out);
    prof_mark(e, nm, 2.0 * M * (double)cproj.out * cproj.in + 4.0 * M * (double)fc1.out * fc1.in,
              2.0 * (double)cproj.out * cproj.in + 4.0 * (double)fc1.out * fc1.in +
                  (double)M * fc1.in * (2.0 + 4.0 + 4.0 + 2.0), s);
  } else {
    e->launches++;
  }
  return cproj_mlp_resid_ln(o, cproj.w, cproj.b, x, norm2.w, norm2.b, fc1.w, fc1.b, fc2.w, fc2.b, ln.w, ln.b, h_out, M,
                            fc1.in, fc1.out, 1e-6f, s);
}
static int L_resid_ln(vited_engine* e, float* x, const act_t* delta, const float* gsrc, const int* gidx, int n_src,
                      const LNorm* ln, act_t* h, int n_seq, int has_cls, int write_x, cudaStream_t s, int g_off = 0) {
  ResidLnArgs a;
  a.x = x; a.delta = delta; a.gather_src = gsrc; a.gather_idx = gidx; a.gather_off = g_off; a.n_src_seq = n_src;
  a.ln_w = ln ? ln->w : nullptr; a.ln_b = ln ? ln->b : nullptr; a.h = h;
  a.n_seq = n_seq; a.n_patch = e->Ne; a.has_cls = has_cls; a.D = e->D; a.write_x = write_x; a.eps = 1e-6f;
  {
    const double rows = (double)n_seq * (e->Ne + (has_cls ? 1 : 0));
    const double per_row = e->D * (4.0 + (delta ? 2.0 : 0.0) + (write_x ? 4.0 : 0.0) + (ln ? 2.0 : 0.0));
    prof_mark(e, "resid_ln", 0.0, rows * per_row, s);
  }
  return resid_ln(a, s);
}
static int L_attn_self(vited_engine* e, const act_t* qkv, act_t* o, int n_seq, int has_cls, cudaStream_t s) {
  AttnArgs a;
  const int D = e->D;
  a.q = qkv; a.q_ld = 3 * D; a.k = qkv + D; a.k_ld = 3 * D; a.v = qkv + 2 * D; a.v_ld = 3 * D; a.o = o; a.o_ld = D;
  a.n_seq = n_seq; a.n_heads = e->H; a.head_dim = e->hd;
  a.nq_patch = e->Ne; a.q_has_cls = has_cls; a.nk_patch = e->Ne; a.k_has_cls = has_cls;
  a.n_kv_seq = n_seq; a.kv_index = nullptr; a.scale = e->scale;
  {
    const double n = e->Ne + (has_cls ? 1 : 0);
    prof_mark(e, "attn_self", 4.0 * n_seq * n * n * e->D, (double)n_seq * n * e->D * 2.0 * 4.0, s);
  }
  return attention(a, e->attn_impl, s);
}
static int L_attn_cross(vited_engine* e, const act_t* q, const act_t* kv, act_t* o, int n_seq, int n_kv_seq,
                        const int* kv_index, cudaStream_t s) {
  AttnArgs a;
  const int D = e->D;
  a.q = q; a.q_ld = D; a.k = kv; a.k_ld = 2 * D; a.v = kv + D; a.v_ld = 2 * D; a.o = o; a.o_ld = D;
  a.n_seq = n_seq; a.n_heads = e->H; a.head_dim = e->hd;
  a.nq_patch = e->Ne; a.q_has_cls = 1; a.nk_patch = e->Ne; a.k_has_cls = 0;
  a.n_kv_seq = n_kv_seq; a.kv_index = kv_index; a.scale = e->scale;
  prof_mark(e, "attn_cross", 4.0 * n_seq * (double)e->Nd * e->Ne * e->D, (double)n_seq * e->Nd * e->D * 2.0 * 2.0, s);
  return attention(a, e->attn_impl, s);
}

// class-token-only attention (last decoder layer). q/o are the full split-layout buffers: only their class-token rows
// (row n_seq*Ne + b) are read / written.
static int L_attn_cls(vited_engine* e, const act_t* q, int q_ld, const act_t* k, const act_t* v, int kv_ld, act_t* o,
                      int n_seq, int k_has_cls, int n_kv_seq, const int* kv_index, cudaStream_t s) {
  AttnArgs a;
  a.q = q; a.q_ld = q_ld; a.k = k; a.k_ld = kv_ld; a.v = v; a.v_ld = kv_ld; a.o = o; a.o_ld = e->D;
  a.n_seq = n_seq; a.n_heads = e->H; a.head_dim = e->hd;
  a.nq_patch = e->Ne; a.q_has_cls = 1; a.nk_patch = e->Ne; a.k_has_cls = k_has_cls;
  a.n_kv_seq = n_kv_seq; a.kv_index = kv_index; a.scale = e->scale;
  prof_mark(e, "attn_cls", 4.0 * n_seq * (double)(e->Ne + k_has_cls) * e->D,
            (double)n_seq * (e->Ne + k_has_cls) * e->D * 2.0 * 2.0, s);
  return attention_cls(a, s);
}
// resid_ln over a plain block of `rows` rows (no split-layout bookkeeping): used for the class-token rows alone
static int L_resid_ln_rows(vited_engine* e, float* x, const act_t* delta, const float* gsrc_cls_rows, const int* gidx,
                           const LNorm* ln, act_t* h, int rows, cudaStream_t s, int g_off = 0) {
  ResidLnArgs a;
  a.x = x; a.delta = delta; a.gather_src = gsrc_cls_rows; a.gather_idx = gidx; a.gather_off = g_off; a.n_src_seq = 0;
  a.ln_w = ln ? ln->w : nullptr; a.ln_b = ln ? ln->b : nullptr; a.h = h;
  a.n_seq = rows; a.n_patch = 1; a.has_cls = 0; a.D = e->D; a.write_x = 1; a.eps = 1e-6f;
  prof_mark(e, "resid_ln", 0.0, (double)rows * e->D * 12.0, s);
  return resid_ln(a, s);
}

static int ensure_rows(vited_engine* e, size_t rows) {
  const size_t D = e->D;
  TRY(e->x.ensure(rows * D * 4));
  TRY(e->h.ensure(rows * D * 2));
  TRY(e->qkv.ensure(rows * 3 * D * 2));
  TRY(e->o.ensure(rows * D * 2));
  TRY(e->q.ensure(rows * D * 2));
  TRY(e->delta.ensure(rows * D * 2));
  TRY(e->hid.ensure(rows * (size_t)e->hidden * 2));
  return 0;
}

// Every entry point makes the engine's device current for its own duration and puts the caller's device back on return
// (the caller -- PyTorch -- tracks its own current device and must not find it changed underneath it).
struct DeviceScope {
  int prev = -1;
  explicit DeviceScope(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    if (prev != dev) cudaSetDevice(dev); else prev = -1;
  }
  ~DeviceScope() { if (prev >= 0) cudaSetDevice(prev); }
  DeviceScope(const DeviceScope&) = delete;
  DeviceScope& operator=(const DeviceScope&) = delete;
};

static int check_ready(vited_engine* e) {
  VITED_CHECK(e != nullptr, "null engine");
  VITED_CHECK(e->loaded == (int)e->names.size(), "weights not loaded: %d of %d state_dict tensors received", e->loaded,
              (int)e->names.size());
  return 0;
}

// items per sub-batch so that token rows stay near chunk_rows
static int items_per_batch(vited_engine* e) {
  int64_t n = e->chunk_rows / e->Nd;
  return (int)(n < 1 ? 1 : n);
}

// patch tokens of B images -> e->tok (fp16 [B*Ne, D]); img_stride = elements between consecutive images.
// `u8`: the images are [B, S, S, in_chans] bytes (ToTensor + Normalize(.5, .5) applied on the way, im2col_u8_patches),
// otherwise [B, in_chans, S, S] fp32. `items` (device, [B]) non-null: image b is images[items[b]] of a contiguous set.
static int patch_tokens(vited_engine* e, const void* images, bool u8, size_t img_stride, int B, cudaStream_t s,
                        const int* items = nullptr) {
  const vited_config& c = e->cfg;
  const size_t rows = (size_t)B * e->Ne;
  TRY(e->col.ensure(rows * e->Kpe * 2));
  TRY(e->tok.ensure(rows * e->D * 2));
  const size_t img_elems = (size_t)c.in_chans * c.img_size * c.img_size;
  if (u8) {
    VITED_CHECK(img_stride == img_elems, "patch_tokens: uint8 images must be contiguous");
    prof_mark(e, "im2col_u8", 0.0, (double)rows * e->Kpe * 3.0, s);
    TRY(im2col_u8_patches(static_cast<const uint8_t*>(images), e->col.as<act_t>(), B, c.in_chans, c.img_size,
                          c.patch_size, s, items));
  } else if (img_stride == img_elems) {
    prof_mark(e, "im2col", 0.0, (double)rows * e->Kpe * 6.0, s);
    TRY(im2col_patches(static_cast<const float*>(images), e->col.as<act_t>(), B, c.in_chans, c.img_size, c.patch_size, s,
                       items));
  } else {
    VITED_CHECK(items == nullptr, "patch_tokens: gathered images must be contiguous");
    for (int b = 0; b < B; ++b) {
      prof_mark(e, "im2col", 0.0, (double)e->Ne * e->Kpe * 6.0, s);
      TRY(im2col_patches(static_cast<const float*>(images) + (size_t)b * img_stride,
                         e->col.as<act_t>() + (size_t)b * e->Ne * e->Kpe, 1, c.in_chans, c.img_size, c.patch_size, s));
    }
  }
  TRY(L_gemm(e, e->col.as<act_t>(), e->patch, e->tok.as<act_t>(), (int)rows, ACT_NONE, s));
  return 0;
}

// forward_first_part (vision_transformer.py:382-388) for a sub-batch whose patch tokens are in e->tok.
static int encoder_stack(vited_engine* e, int B, float* out_tokens, cudaStream_t s) {
  const size_t rows = (size_t)B * e->Ne;
  TRY(ensure_rows(e, rows));
  float* x = e->x.as<float>();
  act_t* h = e->h.as<act_t>();
  act_t* delta = e->delta.as<act_t>();
  prof_mark(e, "assemble", 0.0, (double)rows * e->D * 6.0, s);
  TRY(assemble_tokens(e->tok.as<act_t>(), e->pos, e->cls, x, B, e->Ne, e->D, 0, s));
  for (size_t l = 0; l < e->enc.size(); ++l) {
    EncBlock& b = e->enc[l];
    TRY(L_resid_ln(e, x, l == 0 ? nullptr : delta, nullptr, nullptr, 0, &b.norm1, h, B, 0, l == 0 ? 0 : 1, s));
    TRY(L_gemm(e, h, b.qkv, e->qkv.as<act_t>(), (int)rows, ACT_NONE, s));
    TRY(L_attn_self(e, e->qkv.as<act_t>(), e->o.as<act_t>(), B, 0, s));
    TRY(L_gemm(e, e->o.as<act_t>(), b.proj, delta, (int)rows, ACT_NONE, s));
    TRY(L_resid_ln(e, x, delta, nullptr, nullptr, 0, &b.norm2, h, B, 0, 1, s));
    TRY(L_gemm(e, h, b.fc1, e->hid.as<act_t>(), (int)rows, ACT_GELU, s));
    TRY(L_gemm(e, e->hid.as<act_t>(), b.fc2, delta, (int)rows, ACT_NONE, s));
  }
  prof_mark(e, "add_delta_out", 0.0, (double)rows * e->D * 10.0, s);
  TRY(add_delta_out(x, delta, out_tokens, rows, e->D, s));
  return 0;
}

// prepare_x2 (vision_transformer.py:390-395) [+ decoder layer 0's self-attention sub-block when cached] for a
// sub-batch whose patch tokens are in e->tok. Result (split layout, B sequences) is left in e->x.
static int decoder_item_state(vited_engine* e, int B, cudaStream_t s) {
  const size_t rows = (size_t)B * e->Nd;
  TRY(ensure_rows(e, rows));
  float* x = e->x.as<float>();
  prof_mark(e, "assemble", 0.0, (double)rows * e->D * 6.0, s);
  TRY(assemble_tokens(e->tok.as<act_t>(), e->pos, e->cls, x, B, e->Ne, e->D, 1, s));
  if (e->cache_layer0) {
    DecBlock& b = e->dec[0];
    TRY(L_resid_ln(e, x, nullptr, nullptr, nullptr, 0, &b.norm1, e->h.as<act_t>(), B, 1, 0, s));
    TRY(L_gemm(e, e->h.as<act_t>(), b.qkv, e->qkv.as<act_t>(), (int)rows, ACT_NONE, s));
    TRY(L_attn_self(e, e->qkv.as<act_t>(), e->o.as<act_t>(), B, 1, s));
    TRY(L_gemm(e, e->o.as<act_t>(), b.proj, e->delta.as<act_t>(), (int)rows, ACT_NONE, s));
    TRY(L_resid_ln(e, x, e->delta.as<act_t>(), nullptr, nullptr, 0, nullptr, nullptr, B, 1, 1, s));
  }
  return 0;
}

// copy a sub-batch in split layout (B sequences in e->x) into rows [i0, i0+B) of a split-layout buffer of N sequences
static int scatter_split(vited_engine* e, float* dst, int N, int i0, int B, cudaStream_t s) {
  const size_t D = e->D, Ne = e->Ne;
  const float* x = e->x.as<float>();
  if (e->profile) { prof_mark(e, "copy", 0.0, (double)B * (Ne + 1) * D * 8.0, s); e->launches--; }
  VITED_CUDA_OK(cudaMemcpyAsync(dst + (size_t)i0 * Ne * D, x, (size_t)B * Ne * D * 4, cudaMemcpyDeviceToDevice, s));
  VITED_CUDA_OK(cudaMemcpyAsync(dst + ((size_t)N * Ne + i0) * D, x + (size_t)B * Ne * D, (size_t)B * D * 4,
                                cudaMemcpyDeviceToDevice, s));
  return 0;
}

// kv(norm_context(ctx)) for every decoder layer (vision_transformer.py:270, :178): ctx [n*Ne, D] f32 ->
// e->kv, layer l at offset l * n*Ne*2D (fp16)
static int build_kv(vited_engine* e, const float* ctx, int n, cudaStream_t s) {
  const size_t rows = (size_t)n * e->Ne;
  const size_t per_layer = rows * 2 * e->D;
  TRY(e->kv.ensure(per_layer * e->dec.size() * 2));
  TRY(e->h.ensure(rows * e->D * 2));
  for (size_t l = 0; l < e->dec.size(); ++l) {
    DecBlock& b = e->dec[l];
    TRY(L_resid_ln(e, const_cast<float*>(ctx), nullptr, nullptr, nullptr, 0, &b.norm_context, e->h.as<act_t>(), n, 0, 0,
                   s));
    TRY(L_gemm(e, e->h.as<act_t>(), b.kv, e->kv.as<act_t>() + l * per_layer, (int)rows, ACT_NONE, s));
  }
  return 0;
}

// cross_part + head (vision_transformer.py:397-401, :415-417) for P pairs.
//   ci[p]: context sequence inside the current KV block; xj[p]: item whose decoder state seeds the pair.
//   xsrc holds the decoder input states of items [x_off, x_off + n_src) in split layout.
static int decode_chunk(vited_engine* e, int P, const int* ci, const int* xj, const float* xsrc, int n_src, int x_off,
                        int n_kv_seq, HeadArgs head, cudaStream_t s) {
  const size_t rows = (size_t)P * e->Nd;
  TRY(ensure_rows(e, rows));
  const size_t D = e->D;
  const size_t cls_off = (size_t)P * e->Ne;      // first class-token row in every [rows, *] buffer
  float* x = e->x.as<float>();
  act_t* h = e->h.as<act_t>();
  act_t* delta = e->delta.as<act_t>();
  act_t* qkv = e->qkv.as<act_t>();
  act_t* o = e->o.as<act_t>();
  act_t* q = e->q.as<act_t>();
  act_t* hid = e->hid.as<act_t>();
  const size_t kv_per_layer = (size_t)n_kv_seq * e->Ne * 2 * D;
  const size_t L = e->dec.size();
  // With FUSE_LN the residual add + LayerNorm of a sub-block boundary runs in the epilogue of the GEMM that produces
  // the sub-block output (proj -> norm_cross, cross proj -> norm2, fc2 -> the NEXT layer's norm1), so `delta` is never
  // written and the separate resid_ln pass disappears.
  const bool fuse = use_fused_ln(e, rows, e->dec[0].proj);
  bool h_is_norm1 = false;   // h already holds norm1(x) of the current layer (fc2 of the previous layer was fused)
  for (size_t l = 0; l < L; ++l) {
    DecBlock& b = e->dec[l];
    const bool first = (l == 0);
    // In the last layer only row 0 (the class token) of every sequence reaches the head, so after the keys/values of
    // its self-attention are formed every kernel runs on the P class-token rows alone.
    const bool tail = e->prune_tail && (l + 1 == L);
    const act_t* kvl = e->kv.as<act_t>() + l * kv_per_layer;
    if (!tail) {
      if (first && e->cache_layer0) {
        TRY(L_resid_ln(e, x, nullptr, xsrc, xj, n_src, &b.norm_cross, h, P, 1, 1, s, x_off));
      } else {
        if (first) TRY(L_resid_ln(e, x, nullptr, xsrc, xj, n_src, &b.norm1, h, P, 1, 1, s, x_off));
        else if (!h_is_norm1) TRY(L_resid_ln(e, x, delta, nullptr, nullptr, 0, &b.norm1, h, P, 1, 1, s));
        TRY(L_gemm(e, h, b.qkv, qkv, (int)rows, ACT_NONE, s));
        TRY(L_attn_self(e, qkv, o, P, 1, s));
        if (fuse) {
          TRY(L_gemm_ln(e, o, b.proj, x, b.norm_cross, h, (int)rows, s));
        } else {
          TRY(L_gemm(e, o, b.proj, delta, (int)rows, ACT_NONE, s));
          TRY(L_resid_ln(e, x, delta, nullptr, nullptr, 0, &b.norm_cross, h, P, 1, 1, s));
        }
      }
      TRY(L_gemm(e, h, b.q, q, (int)rows, ACT_NONE, s));
      TRY(L_attn_cross(e, q, kvl, o, P, n_kv_seq, ci, s));
      h_is_norm1 = false;
      if (fuse && l + 1 < L && use_fused_mlp(e, rows, b.cproj, b.fc1, b.fc2)) {
        // the cross projection, its residual add and norm2, the whole MLP sub-block, its residual add and the next
        // layer's norm1 in one kernel: neither the intermediate residual rows nor norm2's output nor `hid` is written
        TRY(L_cproj_mlp_ln(e, o, b.cproj, b.norm2, b.fc1, b.fc2, x, e->dec[l + 1].norm1, h, (int)rows, s));
        h_is_norm1 = true;
      } else {
        if (fuse) {
          TRY(L_gemm_ln(e, o, b.cproj, x, b.norm2, h, (int)rows, s));
        } else {
          TRY(L_gemm(e, o, b.cproj, delta, (int)rows, ACT_NONE, s));
          TRY(L_resid_ln(e, x, delta, nullptr, nullptr, 0, &b.norm2, h, P, 1, 1, s));
        }
        if (fuse && l + 1 < L) {
          TRY(L_gemm(e, h, b.fc1, hid, (int)rows, ACT_GELU, s));
          TRY(L_gemm_ln(e, hid, b.fc2, x, e->dec[l + 1].norm1, h, (int)rows, s));
          h_is_norm1 = true;
        } else {
          TRY(L_gemm(e, h, b.fc1, hid, (int)rows, ACT_GELU, s));
          TRY(L_gemm(e, hid, b.fc2, delta, (int)rows, ACT_NONE, s));
        }
      }
    } else {
      float* x_c = x + cls_off * D;
      act_t* h_c = h + cls_off * D;
      act_t* d_c = delta + cls_off * D;
      act_t* q_c = q + cls_off * D;
      act_t* o_c = o + cls_off * D;
      if (first && e->cache_layer0) {
        // single-layer decoder with the layer-0 cache: gather the class-token rows only
        TRY(L_resid_ln_rows(e, x_c, nullptr, xsrc + (size_t)n_src * e->Ne * D, xj, &b.norm_cross, h_c, P, s, x_off));
      } else {
        if (first) TRY(L_resid_ln(e, x, nullptr, xsrc, xj, n_src, &b.norm1, h, P, 1, 1, s, x_off));
        else if (!h_is_norm1) TRY(L_resid_ln(e, x, delta, nullptr, nullptr, 0, &b.norm1, h, P, 1, 1, s));
        // keys/values for every token, the query for the class token only (qkv rows: [0,D) q, [D,3D) k|v)
        Linear w_kv = b.qkv; w_kv.w = b.qkv.w + D * D; w_kv.b = b.qkv.b + D; w_kv.out = 2 * (int)D;
        Linear w_q = b.qkv; w_q.out = (int)D;
        TRY(L_gemm(e, h, w_kv, qkv, (int)rows, ACT_NONE, s));          // [rows, 2D]
        TRY(L_gemm(e, h_c, w_q, q_c, P, ACT_NONE, s));                 // [P, D]
        TRY(L_attn_cls(e, q, (int)D, qkv, qkv + D, 2 * (int)D, o, P, 1, P, nullptr, s));
        TRY(L_gemm(e, o_c, b.proj, d_c, P, ACT_NONE, s));
        TRY(L_resid_ln_rows(e, x_c, d_c, nullptr, nullptr, &b.norm_cross, h_c, P, s));
      }
      TRY(L_gemm(e, h_c, b.q, q_c, P, ACT_NONE, s));
      TRY(L_attn_cls(e, q, (int)D, kvl, kvl + D, 2 * (int)D, o, P, 0, n_kv_seq, ci, s));
      TRY(L_gemm(e, o_c, b.cproj, d_c, P, ACT_NONE, s));
      TRY(L_resid_ln_rows(e, x_c, d_c, nullptr, nullptr, &b.norm2, h_c, P, s));
      TRY(L_gemm(e, h_c, b.fc1, hid, P, ACT_GELU, s));
      TRY(L_gemm(e, hid, b.fc2, d_c, P, ACT_NONE, s));
      h_is_norm1 = false;
    }
  }
  head.x = x + cls_off * D;
  head.delta = delta + cls_off * D;
  head.ln_w = e->norm.w; head.ln_b = e->norm.b; head.head_w = e->head_w; head.head_b = e->head_b;
  head.P = P; head.D = e->D; head.C = e->C; head.eps = 1e-6f;
  prof_mark(e, "head", 0.0, (double)P * e->D * 6.0, s);
  TRY(head_logits(head, s));
  return 0;
}

// pair list of grid rows [r0, r1) x columns [ca, cb) into e->ci / e->xj (generated on the device; nothing to upload or wait for)
static int build_pair_list(vited_engine* e, int mode, int r0, int r1, int ca, int cb, size_t* total, cudaStream_t s) {
  *total = pair_list_count(mode, r0, r1, ca, cb);
  if (*total == 0) return 0;
  TRY(e->ci.ensure(*total * sizeof(int) + 16));
  TRY(e->xj.ensure(*total * sizeof(int) + 16));
  prof_mark(e, "pair_list", 0.0, (double)*total * 8.0, s);
  return pair_list(mode, r0, r1, ca, cb, e->ci.as<int>(), e->xj.as<int>(), s);
}

}  // namespace vited

// =====================================================================================================================
// C-ABI
// =====================================================================================================================
namespace vited {
bool pdl_enabled() {
  static const int on = [] { const char* v = getenv("VITED_PDL"); return v == nullptr ? 0 : atoi(v); }();
  return on != 0;
}
}  // namespace vited

extern "C" {

const char* vited_last_error(void) { return get_error(); }

int vited_create(const vited_config* cfg, int device, vited_engine** out) {
  VITED_CHECK(cfg != nullptr && out != nullptr, "vited_create: null argument");
  int ndev = 0;
  cudaError_t ce = cudaGetDeviceCount(&ndev);
  VITED_CHECK(ce == cudaSuccess && ndev > 0, "vited_create: no CUDA device available (%s); this path has no CPU fallback",
              cudaGetErrorString(ce));
  VITED_CHECK(device >= 0 && device < ndev, "vited_create: device %d out of range (%d devices)", device, ndev);
  DeviceScope scope(device);
  cudaDeviceProp prop;
  VITED_CUDA_OK(cudaGetDeviceProperties(&prop, device));
  VITED_CHECK(prop.major == 10, "vited_create: device %d is sm_%d%d; this library contains sm_100a code only", device,
              prop.major, prop.minor);
  vited_engine* e = new vited_engine();
  e->cfg = *cfg;
  e->device = device;
  const char* cr = getenv("VITED_CHUNK_ROWS");
  if (cr && atoll(cr) > 0) e->chunk_rows = atoll(cr);
  const char* fm = getenv("VITED_FUSE_MLP");   // A/B runs of bench.py; vited_set_option(VITED_OPT_FUSE_MLP) is the API
  if (fm) e->fuse_mlp = atoi(fm) ? 1 : 0;
  if (build(e) != 0) {
    vited_destroy(e);
    return 1;
  }
  *out = e;
  return 0;
}

void vited_destroy(vited_engine* e) {
  if (!e) return;
  DeviceScope scope(e->device);
  cudaDeviceSynchronize();
  for (void* p : e->owned) cudaFree(p);
  DevBuf* bufs[] = {&e->x, &e->h, &e->qkv, &e->o, &e->q, &e->delta, &e->hid, &e->col, &e->tok, &e->xsrc, &e->enc_tok,
                    &e->kv, &e->ci, &e->xj, &e->tmp_tok, &e->out_pos, &e->pl_items, &e->pl_hist, &e->pl_info};
  for (DevBuf* b : bufs) b->release();
  for (cudaEvent_t ev : e->ev_pool) cudaEventDestroy(ev);
  delete e;
}

int vited_set_option(vited_engine* e, int option, int64_t value) {
  VITED_CHECK(e != nullptr, "null engine");
  switch (option) {
    case VITED_OPT_GEMM_IMPL: e->gemm_impl = value ? IMPL_REF : IMPL_FAST; return 0;
    case VITED_OPT_ATTN_IMPL: e->attn_impl = value == 1 ? IMPL_REF : value == 2 ? IMPL_MMA_SYNC : IMPL_FAST; return 0;
    case VITED_OPT_CHUNK_ROWS:
      VITED_CHECK(value >= 1, "chunk_rows must be positive");
      e->chunk_rows = value;
      return 0;
    case VITED_OPT_CACHE_LAYER0: e->cache_layer0 = value ? 1 : 0; return 0;
    case VITED_OPT_PRUNE_TAIL: e->prune_tail = value ? 1 : 0; return 0;
    case VITED_OPT_FUSE_LN: e->fuse_ln = value ? 1 : 0; return 0;
    case VITED_OPT_FUSE_MLP: e->fuse_mlp = value ? 1 : 0; return 0;
    case VITED_OPT_KV_BUDGET_MB:
      VITED_CHECK(value >= 1, "kv budget must be positive");
      e->kv_budget_mb = value;
      return 0;
    case VITED_OPT_XSRC_BUDGET_MB:
      VITED_CHECK(value >= 1, "column state budget must be positive");
      e->xsrc_budget_mb = value;
      return 0;
    case VITED_OPT_PROFILE:
      e->profile = value ? 1 : 0;
      e->recs.clear();
      e->ev_used = 0;
      return 0;
    default: set_error("unknown option %d", option); return 1;
  }
}

int vited_load_weight(vited_engine* e, const char* name, const float* data, int64_t numel, void* stream) {
  VITED_CHECK(e != nullptr && name != nullptr && data != nullptr, "vited_load_weight: null argument");
  DeviceScope scope(e->device);
  auto it = e->slots.find(name);
  VITED_CHECK(it != e->slots.end(), "unexpected key in state_dict: %s", name);
  Slot& sl = it->second;
  VITED_CHECK(sl.numel == numel, "size mismatch for %s: expected %lld elements, got %lld", name, (long long)sl.numel,
              (long long)numel);
  cudaStream_t s = (cudaStream_t)stream;
  if (sl.to_act) {
    TRY(f32_to_act(data, reinterpret_cast<act_t*>(sl.dst), (size_t)numel, s));
  } else {
    VITED_CUDA_OK(cudaMemcpyAsync(sl.dst, data, (size_t)numel * 4, cudaMemcpyDeviceToDevice, s));
  }
  VITED_CUDA_OK(cudaStreamSynchronize(s));
  if (!sl.loaded) {
    sl.loaded = true;
    e->loaded++;
  }
  return 0;
}

int vited_num_weights_expected(vited_engine* e) { return e ? (int)e->names.size() : 0; }
int vited_num_weights_loaded(vited_engine* e) { return e ? e->loaded : 0; }
const char* vited_weight_name(vited_engine* e, int i) {
  if (!e || i < 0 || i >= (int)e->names.size()) return nullptr;
  return e->names[i].c_str();
}

int vited_encode(vited_engine* e, const float* images, int B, float* out_tokens, void* stream) {
  TRY(check_ready(e));
  DeviceScope scope(e->device);
  VITED_CHECK(B >= 0 && (B == 0 || (images && out_tokens)), "vited_encode: bad arguments");
  cudaStream_t s = (cudaStream_t)stream;
  const size_t img = (size_t)e->cfg.in_chans * e->cfg.img_size * e->cfg.img_size;
  const int step = items_per_batch(e);
  for (int i0 = 0; i0 < B; i0 += step) {
    const int n = (B - i0 < step) ? (B - i0) : step;
    TRY(patch_tokens(e, images + (size_t)i0 * img, false, img, n, s));
    TRY(encoder_stack(e, n, out_tokens + (size_t)i0 * e->Ne * e->D, s));
  }
  return 0;
}

static int decode_impl(vited_engine* e, const float* ctx_tokens, const float* images, size_t img_stride, int B,
                       float* out_logits, cudaStream_t s) {
  const int step = items_per_batch(e);
  for (int i0 = 0; i0 < B; i0 += step) {
    const int n = (B - i0 < step) ? (B - i0) : step;
    // decoder input state of the n x2 images
    TRY(patch_tokens(e, images + (size_t)i0 * img_stride, false, img_stride, n, s));
    TRY(decoder_item_state(e, n, s));
    TRY(e->xsrc.ensure((size_t)n * e->Nd * e->D * 4));
    VITED_CUDA_OK(cudaMemcpyAsync(e->xsrc.p, e->x.p, (size_t)n * e->Nd * e->D * 4, cudaMemcpyDeviceToDevice, s));
    TRY(build_kv(e, ctx_tokens + (size_t)i0 * e->Ne * e->D, n, s));
    size_t total = 0;
    TRY(build_pair_list(e, 2, 0, n, 0, n, &total, s));   // pair p: context p, decoder state p
    HeadArgs head = {};
    head.out = out_logits + (size_t)i0 * e->C;
    head.ci = nullptr; head.xj = nullptr; head.row_begin = 0; head.n_items = 0;
    TRY(decode_chunk(e, n, e->ci.as<int>(), e->xj.as<int>(), e->xsrc.as<float>(), n, 0, n, head, s));
  }
  return 0;
}

int vited_decode(vited_engine* e, const float* ctx_tokens, const float* images, int B, float* out_logits,
                 void* stream) {
  TRY(check_ready(e));
  DeviceScope scope(e->device);
  VITED_CHECK(B >= 0 && (B == 0 || (ctx_tokens && images && out_logits)), "vited_decode: bad arguments");
  const size_t img = (size_t)e->cfg.in_chans * e->cfg.img_size * e->cfg.img_size;
  return decode_impl(e, ctx_tokens, images, img, B, out_logits, (cudaStream_t)stream);
}

int vited_forward_pairs(vited_engine* e, const float* pairs, int B, float* out_logits, void* stream) {
  TRY(check_ready(e));
  DeviceScope scope(e->device);
  VITED_CHECK(B >= 0 && (B == 0 || (pairs && out_logits)), "vited_forward_pairs: bad arguments");
  cudaStream_t s = (cudaStream_t)stream;
  const size_t img = (size_t)e->cfg.in_chans * e->cfg.img_size * e->cfg.img_size;
  const int step = items_per_batch(e);
  for (int i0 = 0; i0 < B; i0 += step) {
    const int n = (B - i0 < step) ? (B - i0) : step;
    const float* base = pairs + (size_t)i0 * 2 * img;
    TRY(e->tmp_tok.ensure((size_t)n * e->Ne * e->D * 4));
    TRY(patch_tokens(e, base, false, 2 * img, n, s));            // x1 = pairs[:, 0]
    TRY(encoder_stack(e, n, e->tmp_tok.as<float>(), s));
    TRY(decode_impl(e, e->tmp_tok.as<float>(), base + img, 2 * img, n, out_logits + (size_t)i0 * e->C, s));  // x2 = pairs[:, 1]
  }
  return 0;
}

// decoder input states of items [ca, cb) -> e->xsrc (split layout, cb - ca sequences). `items` non-null: of items
// items[ca .. cb) (device list) instead.
static int build_xsrc(vited_engine* e, const char* images, bool u8, size_t img_bytes, int ca, int cb, bool headroom,
                      cudaStream_t s, const int* items = nullptr) {
  const int n_src = cb - ca;
  const size_t img = (size_t)e->cfg.in_chans * e->cfg.img_size * e->cfg.img_size;
  const int step = items_per_batch(e);
  TRY(e->xsrc.ensure((size_t)n_src * e->Nd * e->D * 4, headroom));
  for (int i0 = 0; i0 < n_src; i0 += step) {
    const int n = (n_src - i0 < step) ? (n_src - i0) : step;
    if (items) TRY(patch_tokens(e, images, u8, img, n, s, items + ca + i0));
    else TRY(patch_tokens(e, images + (size_t)(ca + i0) * img_bytes, u8, img, n, s));
    TRY(decoder_item_state(e, n, s));
    TRY(scatter_split(e, e->xsrc.as<float>(), n_src, i0, n, s));
  }
  return 0;
}

// items whose decoder input states fit OPT_XSRC_BUDGET_MB (columns per window), at least one
static int64_t xsrc_window_items(vited_engine* e) {
  const int64_t cw = (int64_t)((size_t)e->xsrc_budget_mb * 1000000 / ((size_t)e->Nd * e->D * 4));
  return cw < 1 ? 1 : cw;
}
// context items whose K/V cache (every decoder layer) fits OPT_KV_BUDGET_MB, at least one
static int kv_block_items(vited_engine* e) {
  const int rb = (int)((size_t)e->kv_budget_mb * 1000000 / (e->dec.size() * e->Ne * 2 * e->D * 2));
  return rb < 1 ? 1 : rb;
}

// vited_score_grid / vited_score_grid_u8: one grid loop for both image formats
static int score_grid_impl(vited_engine* e, const void* images_in, bool u8, int N, int mode, int row_begin, int row_end,
                           float* out, cudaStream_t s) {
  TRY(check_ready(e));
  DeviceScope scope(e->device);
  VITED_CHECK(mode == VITED_GRID_ORDERED_OFFDIAG || mode == VITED_GRID_UPPER_TRI_DIAG, "unknown grid mode %d", mode);
  VITED_CHECK(N >= 0 && row_begin >= 0 && row_begin <= row_end && row_end <= N, "bad row range [%d, %d) for N=%d",
              row_begin, row_end, N);
  if (N == 0 || row_begin == row_end) return 0;
  VITED_CHECK(images_in && out, "vited_score_grid: null pointer");
  const char* images = static_cast<const char*>(images_in);
  const size_t img = (size_t)e->cfg.in_chans * e->cfg.img_size * e->cfg.img_size;
  const size_t img_bytes = img * (u8 ? 1 : 4);
  const size_t D = e->D, Ne = e->Ne;
  const int step = items_per_batch(e);
  const int pair_mode = mode == VITED_GRID_ORDERED_OFFDIAG ? 0 : 1;

  // 1) decoder input state of every item that appears as a COLUMN of this row shard: computed once per item, reused
  //    by every pair. The upper-triangular grid (hisfrag.py:166-167) never pairs a row with a column j < row_begin,
  //    so a row shard builds (and holds) only the states of items [row_begin, N). When those states exceed the
  //    budget (default 32 GB: 20,345 Hisfrag items at 1.57 MB), they are built per column window of at most the
  //    budget, inside the loop over K/V row blocks below; otherwise once, here, for the whole call.
  const int c0 = (mode == VITED_GRID_UPPER_TRI_DIAG) ? row_begin : 0;
  const int n_cols = N - c0;
  const int64_t cw = xsrc_window_items(e);
  const bool one_window = n_cols <= cw;
  const int win = one_window ? n_cols : (int)cw;
  if (one_window) TRY(build_xsrc(e, images, u8, img_bytes, c0, N, true, s));

  // 2) context rows in blocks whose K/V cache stays within the budget (default 8 GB)
  const int rb = kv_block_items(e);
  const int pairs_per_chunk = items_per_batch(e);
  for (int r0 = row_begin; r0 < row_end; r0 += rb) {
    const int r1 = (r0 + rb < row_end) ? (r0 + rb) : row_end;
    const int nr = r1 - r0;
    // encoder tokens of the block's items
    TRY(e->enc_tok.ensure((size_t)nr * Ne * D * 4));
    for (int i0 = 0; i0 < nr; i0 += step) {
      const int n = (nr - i0 < step) ? (nr - i0) : step;
      TRY(patch_tokens(e, images + (size_t)(r0 + i0) * img_bytes, u8, img, n, s));
      TRY(encoder_stack(e, n, e->enc_tok.as<float>() + (size_t)i0 * Ne * D, s));
    }
    TRY(build_kv(e, e->enc_tok.as<float>(), nr, s));
    for (int ca = c0; ca < N; ca += win) {
      const int cb = (ca + win < N) ? (ca + win) : N;
      if (mode == VITED_GRID_UPPER_TRI_DIAG && cb <= r0) continue;   // no column of the window pairs with these rows
      if (!one_window) TRY(build_xsrc(e, images, u8, img_bytes, ca, cb, false, s));
      // pair list of the block x window, i-major (data/datasets/pieces_dataset.py:27-32 / hisfrag.py:166-167)
      size_t total = 0;
      TRY(build_pair_list(e, pair_mode, r0, r1, ca, cb, &total, s));
      if (total == 0) continue;
      // equal chunks: a short last chunk would run every kernel of the stack at a fraction of a wave
      const size_t n_chunks = (total + pairs_per_chunk - 1) / pairs_per_chunk;
      const size_t chunk = (total + n_chunks - 1) / n_chunks;
      for (size_t p0 = 0; p0 < total; p0 += chunk) {
        const int P = (int)((total - p0 < chunk) ? (total - p0) : chunk);
        HeadArgs head = {};
        head.out = out + (size_t)(r0 - row_begin) * N * e->C;
        head.ci = e->ci.as<int>() + p0;
        head.xj = e->xj.as<int>() + p0;
        head.row_begin = 0;  // ci is already relative to r0
        head.n_items = N;
        TRY(decode_chunk(e, P, e->ci.as<int>() + p0, e->xj.as<int>() + p0, e->xsrc.as<float>(), cb - ca, ca, nr, head,
                         s));
      }
    }
  }
  return 0;
}

int vited_score_grid(vited_engine* e, const float* images, int N, int mode, int row_begin, int row_end, float* out,
                     void* stream) {
  return score_grid_impl(e, images, false, N, mode, row_begin, row_end, out, (cudaStream_t)stream);
}

int vited_score_grid_u8(vited_engine* e, const uint8_t* images, int N, int mode, int row_begin, int row_end, float* out,
                        void* stream) {
  return score_grid_impl(e, images, true, N, mode, row_begin, row_end, out, (cudaStream_t)stream);
}

// vited_score_pairs / vited_score_pairs_u8. The distinct context items of the list take the grid's role of rows (slots
// in ascending item order, blocks of kv_block_items), its distinct decoder items that of columns (windows of
// xsrc_window_items); the pairs are bucketed by (block, window) on the device, then the grid's loops run over the cells
// with pairs, with the decoder writing every logit row to the pair's input position.
static int score_pairs_impl(vited_engine* e, const void* images_in, bool u8, int N, const int32_t* pairs,
                            int64_t n_pairs, float* out, cudaStream_t s) {
  TRY(check_ready(e));
  DeviceScope scope(e->device);
  VITED_CHECK(N >= 0, "vited_score_pairs: N = %d", N);
  VITED_CHECK(n_pairs >= 0 && n_pairs <= INT32_MAX, "vited_score_pairs: n_pairs = %lld outside [0, 2^31)",
              (long long)n_pairs);
  if (n_pairs == 0) return 0;
  VITED_CHECK(pairs && out && (images_in || N == 0), "vited_score_pairs: null pointer");
  const int P = (int)n_pairs;
  const char* images = static_cast<const char*>(images_in);
  const size_t img = (size_t)e->cfg.in_chans * e->cfg.img_size * e->cfg.img_size;
  const size_t img_bytes = img * (u8 ? 1 : 4);
  const size_t D = e->D, Ne = e->Ne;
  const int step = items_per_batch(e);

  // cells: at most min(N, P) distinct items on either side
  const int64_t cw = xsrc_window_items(e);
  const int rb = kv_block_items(e);
  const int64_t m = N < P ? N : P;
  const int64_t nw = m > 0 ? (m + cw - 1) / cw : 1;
  const int64_t cells = (m > 0 ? (m + rb - 1) / rb : 1) * nw;
  const int64_t kMaxSortEntries = 1 << 24;
  VITED_CHECK(cells <= kMaxSortEntries,
              "vited_score_pairs: the K/V and decoder-state budgets split %lld items into %lld cells (at most %lld); "
              "raise VITED_OPT_KV_BUDGET_MB / VITED_OPT_XSRC_BUDGET_MB", (long long)m, (long long)cells,
              (long long)kMaxSortEntries);
  // tiles of the counting sort: 1,024 pairs, or more so that the [cells x tiles] histogram stays within 2^24 entries
  int64_t T = 1024;
  if (cells * ((P + T - 1) / T) > kMaxSortEntries) T = ((int64_t)P * cells / kMaxSortEntries + 32) / 32 * 32;
  PairCells pc;
  pc.rb = rb;
  pc.cw = (int)(cw < INT32_MAX ? cw : INT32_MAX);
  pc.nw = (int)nw;
  pc.T = (int)T;
  pc.tiles = (int)((P + T - 1) / T);
  const size_t n_hist = (size_t)cells * pc.tiles;
  const size_t n_info = PL_CELLS + (size_t)cells + 1;
  const size_t Nz = N > 0 ? (size_t)N : 1;
  TRY(e->pl_items.ensure(6 * Nz * sizeof(int)));      // used [2N] | slot [2N] | items [2N]
  TRY(e->pl_hist.ensure(n_hist * sizeof(int)));
  TRY(e->pl_info.ensure(n_info * sizeof(int)));
  TRY(e->ci.ensure((size_t)P * sizeof(int) + 16));
  TRY(e->xj.ensure((size_t)P * sizeof(int) + 16));
  TRY(e->out_pos.ensure((size_t)P * sizeof(int) + 16));
  int* used = e->pl_items.as<int>();
  int* slot = used + 2 * Nz;
  int* items = used + 4 * Nz;
  int* hist = e->pl_hist.as<int>();
  int* info = e->pl_info.as<int>();

  // 1) mark + validate, 2) compact, 3) bucket; 4) one copy back
  VITED_CUDA_OK(cudaMemsetAsync(used, 0, 2 * Nz * sizeof(int), s));
  VITED_CUDA_OK(cudaMemsetAsync(hist, 0, n_hist * sizeof(int), s));
  VITED_CUDA_OK(cudaMemsetAsync(info, 0, n_info * sizeof(int), s));
  VITED_CUDA_OK(cudaMemsetAsync(info + PL_FIRST_BAD, 0xff, sizeof(int), s));
  prof_mark(e, "pair_index", 0.0, (double)P * 8.0, s);
  TRY(pairs_mark(pairs, P, N, used, info, s));
  prof_mark(e, "pair_index", 0.0, (double)Nz * 8.0, s);
  TRY(exclusive_scan(used, slot, N, info + PL_N_CTX, s));
  prof_mark(e, "pair_index", 0.0, (double)Nz * 8.0, s);
  TRY(exclusive_scan(used + Nz, slot + Nz, N, info + PL_N_X2, s));
  prof_mark(e, "pair_index", 0.0, (double)Nz * 16.0, s);
  TRY(pairs_compact(used, slot, items, N, s));
  prof_mark(e, "pair_index", 0.0, (double)P * 16.0 + n_hist * 4.0, s);
  TRY(pairs_bucket_count(pairs, P, N, slot, pc, hist, s));
  prof_mark(e, "pair_index", 0.0, (double)n_hist * 8.0, s);
  TRY(exclusive_scan(hist, hist, (int64_t)n_hist, info + PL_CELLS + cells, s));
  prof_mark(e, "pair_index", 0.0, (double)cells * 8.0, s);
  TRY(pairs_cell_starts(pairs, hist, pc.tiles, (int)cells, info, s));
  prof_mark(e, "pair_index", 0.0, (double)P * 28.0, s);
  TRY(pairs_bucket_scatter(pairs, P, N, slot, pc, hist, e->ci.as<int>(), e->xj.as<int>(), e->out_pos.as<int>(), s));
  std::vector<int> h(n_info);
  VITED_CUDA_OK(cudaMemcpyAsync(h.data(), info, n_info * sizeof(int), cudaMemcpyDeviceToHost, s));
  VITED_CUDA_OK(cudaStreamSynchronize(s));
  VITED_CHECK(h[PL_N_BAD] == 0, "vited_score_pairs: pair %u = (%d, %d) has an index outside [0, %d) (%d such pairs)",
              (unsigned)h[PL_FIRST_BAD], h[PL_BAD_A], h[PL_BAD_B], N, h[PL_N_BAD]);
  const int n_ctx = h[PL_N_CTX], n_x2 = h[PL_N_X2];
  const int* ctx_items = items;
  const int* x2_items = items + Nz;

  // 5) the grid's loops over the cells: K/V blocks outer, decoder-state windows inner
  const bool one_window = n_x2 <= cw;
  if (one_window) TRY(build_xsrc(e, images, u8, img_bytes, 0, n_x2, true, s, x2_items));
  const int pairs_per_chunk = items_per_batch(e);
  for (int blk = 0; (int64_t)blk * rb < n_ctx; ++blk) {
    const int s0 = blk * rb;
    const int nr = (n_ctx - s0 < rb) ? (n_ctx - s0) : rb;
    TRY(e->enc_tok.ensure((size_t)nr * Ne * D * 4));
    for (int i0 = 0; i0 < nr; i0 += step) {
      const int n = (nr - i0 < step) ? (nr - i0) : step;
      TRY(patch_tokens(e, images, u8, img, n, s, ctx_items + s0 + i0));
      TRY(encoder_stack(e, n, e->enc_tok.as<float>() + (size_t)i0 * Ne * D, s));
    }
    TRY(build_kv(e, e->enc_tok.as<float>(), nr, s));
    for (int w = 0; (int64_t)w * cw < n_x2; ++w) {
      const int64_t cell = (int64_t)blk * nw + w;
      const size_t first = (size_t)h[PL_CELLS + cell];
      const size_t total = (size_t)h[PL_CELLS + cell + 1] - first;
      if (total == 0) continue;
      const int ca = (int)(w * cw);
      const int cb = (int)((ca + cw < n_x2) ? (ca + cw) : n_x2);
      if (!one_window) TRY(build_xsrc(e, images, u8, img_bytes, ca, cb, false, s, x2_items));
      // equal chunks, as in score_grid_impl
      const size_t n_chunks = (total + pairs_per_chunk - 1) / pairs_per_chunk;
      const size_t chunk = (total + n_chunks - 1) / n_chunks;
      for (size_t p0 = 0; p0 < total; p0 += chunk) {
        const int Pc = (int)((total - p0 < chunk) ? (total - p0) : chunk);
        HeadArgs head = {};
        head.out = out;
        head.out_pos = e->out_pos.as<int>() + first + p0;
        TRY(decode_chunk(e, Pc, e->ci.as<int>() + first + p0, e->xj.as<int>() + first + p0, e->xsrc.as<float>(),
                         cb - ca, ca, nr, head, s));
      }
    }
  }
  return 0;
}

int vited_score_pairs(vited_engine* e, const float* images, int N, const int32_t* pairs, int64_t n_pairs, float* out,
                      void* stream) {
  return score_pairs_impl(e, images, false, N, pairs, n_pairs, out, (cudaStream_t)stream);
}

int vited_score_pairs_u8(vited_engine* e, const uint8_t* images, int N, const int32_t* pairs, int64_t n_pairs,
                         float* out, void* stream) {
  return score_pairs_impl(e, images, true, N, pairs, n_pairs, out, (cudaStream_t)stream);
}

const char* vited_profile_json(vited_engine* e, void* stream) {
  if (!e) return "{}";
  DeviceScope scope(e->device);
  cudaStream_t s = (cudaStream_t)stream;
  struct Acc { double ms = 0, flops = 0, bytes = 0; long n = 0; };
  std::vector<Acc> acc(e->cls_names.size());
  if (!e->recs.empty()) {
    cudaEvent_t fin;
    cudaEventCreate(&fin);
    cudaEventRecord(fin, s);
    cudaEventSynchronize(fin);
    for (size_t i = 0; i < e->recs.size(); ++i) {
      float ms = 0.f;
      cudaEventElapsedTime(&ms, e->recs[i].ev, i + 1 < e->recs.size() ? e->recs[i + 1].ev : fin);
      Acc& a = acc[e->recs[i].cls];
      a.ms += ms; a.flops += e->recs[i].flops; a.bytes += e->recs[i].bytes; a.n++;
    }
    cudaEventDestroy(fin);
  }
  std::string js = "{";
  bool first = true;
  for (size_t c = 0; c < acc.size(); ++c) {
    if (acc[c].n == 0) continue;
    char buf[256];
    snprintf(buf, sizeof(buf), "%s\"%s\": {\"ms\": %.6f, \"flops\": %.6e, \"bytes\": %.6e, \"launches\": %ld}", first ? "" : ", ",
             e->cls_names[c].c_str(), acc[c].ms, acc[c].flops, acc[c].bytes, acc[c].n);
    js += buf;
    first = false;
  }
  js += "}";
  e->profile_json = js;
  e->recs.clear();
  e->ev_used = 0;
  return e->profile_json.c_str();
}

int64_t vited_launch_count(vited_engine* e) { return e ? e->launches : 0; }
int vited_act_dtype(void) { return VITED_ACT_BF16 ? 1 : 0; }
int64_t vited_workspace_bytes(vited_engine* e) { return e ? e->workspace_bytes() : 0; }

// ---- single-kernel entry points ----
int vited_op_gemm(const void* A, const void* W, const float* bias, void* C, int M, int N, int K, int act, int impl,
                  void* stream) {
  return gemm_act((const act_t*)A, (const act_t*)W, bias, (act_t*)C, M, N, K, act, impl, (cudaStream_t)stream);
}

int vited_op_gemm_resid_ln(const void* A, const void* W, const float* bias, float* x, const float* ln_w,
                           const float* ln_b, void* h, int M, int N, int K, float eps, void* stream) {
  return gemm_resid_ln((const act_t*)A, (const act_t*)W, bias, x, ln_w, ln_b, (act_t*)h, M, N, K, eps, (cudaStream_t)stream);
}

int vited_op_mlp_resid_ln(const void* h_in, const void* W1, const float* b1, const void* W2, const float* b2, float* x,
                          const float* ln_w, const float* ln_b, void* h_out, int M, int D, int hidden, float eps,
                          void* stream) {
  return mlp_resid_ln((const act_t*)h_in, (const act_t*)W1, b1, (const act_t*)W2, b2, x, ln_w, ln_b, (act_t*)h_out, M, D,
                      hidden, eps, (cudaStream_t)stream);
}

int vited_op_cproj_mlp_resid_ln(const void* o, const void* Wp, const float* bp, float* x, const float* ln2_w,
                                const float* ln2_b, const void* W1, const float* b1, const void* W2, const float* b2,
                                const float* ln_w, const float* ln_b, void* h_out, int M, int D, int hidden, float eps,
                                void* stream) {
  return cproj_mlp_resid_ln((const act_t*)o, (const act_t*)Wp, bp, x, ln2_w, ln2_b, (const act_t*)W1, b1,
                            (const act_t*)W2, b2, ln_w, ln_b, (act_t*)h_out, M, D, hidden, eps, (cudaStream_t)stream);
}

int vited_op_resid_ln(float* x, const void* delta, const float* ln_w, const float* ln_b, void* h, int n_seq,
                      int n_patch, int has_cls, int D, float eps, void* stream) {
  ResidLnArgs a;
  a.x = x; a.delta = (const act_t*)delta; a.gather_src = nullptr; a.gather_idx = nullptr; a.n_src_seq = 0;
  a.ln_w = ln_w; a.ln_b = ln_b; a.h = (act_t*)h; a.n_seq = n_seq; a.n_patch = n_patch; a.has_cls = has_cls; a.D = D;
  a.write_x = 1; a.eps = eps;
  return resid_ln(a, (cudaStream_t)stream);
}

int vited_op_attention(const void* q, int q_ld, const void* k, int k_ld, const void* v, int v_ld, void* o, int o_ld,
                       int n_seq, int n_heads, int head_dim, int nq_patch, int q_has_cls, int nk_patch,
                       int k_has_cls, int n_kv_seq, const int32_t* kv_index, float scale, int impl, void* stream) {
  AttnArgs a;
  a.q = (const act_t*)q; a.q_ld = q_ld; a.k = (const act_t*)k; a.k_ld = k_ld; a.v = (const act_t*)v; a.v_ld = v_ld;
  a.o = (act_t*)o; a.o_ld = o_ld; a.n_seq = n_seq; a.n_heads = n_heads; a.head_dim = head_dim;
  a.nq_patch = nq_patch; a.q_has_cls = q_has_cls; a.nk_patch = nk_patch; a.k_has_cls = k_has_cls;
  a.n_kv_seq = n_kv_seq; a.kv_index = kv_index; a.scale = scale;
  return attention(a, impl, (cudaStream_t)stream);
}

int vited_op_attention_cls(const void* q, int q_ld, const void* k, int k_ld, const void* v, int v_ld, void* o, int o_ld,
                           int n_seq, int n_heads, int head_dim, int nk_patch, int k_has_cls, int n_kv_seq,
                           const int32_t* kv_index, float scale, void* stream) {
  // the query side as L_attn_cls passes it: full split-layout buffers of nk_patch patch rows + one class token per sequence
  AttnArgs a;
  a.q = (const act_t*)q; a.q_ld = q_ld; a.k = (const act_t*)k; a.k_ld = k_ld; a.v = (const act_t*)v; a.v_ld = v_ld;
  a.o = (act_t*)o; a.o_ld = o_ld; a.n_seq = n_seq; a.n_heads = n_heads; a.head_dim = head_dim;
  a.nq_patch = nk_patch; a.q_has_cls = 1; a.nk_patch = nk_patch; a.k_has_cls = k_has_cls;
  a.n_kv_seq = n_kv_seq; a.kv_index = kv_index; a.scale = scale;
  return attention_cls(a, (cudaStream_t)stream);
}

int vited_op_head(const float* x, const void* delta, const float* ln_w, const float* ln_b, const float* head_w,
                  const float* head_b, float* out, int P, int D, int C, float eps, void* stream) {
  HeadArgs a = {};
  a.x = x; a.delta = (const act_t*)delta; a.ln_w = ln_w; a.ln_b = ln_b; a.head_w = head_w; a.head_b = head_b;
  a.out = out; a.P = P; a.D = D; a.C = C; a.eps = eps;
  return head_logits(a, (cudaStream_t)stream);
}

int vited_op_im2col(const float* images, void* out, int B, int C, int S, int p, void* stream) {
  return im2col_patches(images, (act_t*)out, B, C, S, p, (cudaStream_t)stream);
}

int vited_op_im2col_u8(const uint8_t* images, void* out, int B, int C, int S, int p, void* stream) {
  return im2col_u8_patches(images, (act_t*)out, B, C, S, p, (cudaStream_t)stream);
}

// ---- training-step kernels (train_ops.cu) ----
int vited_train_cast(const float* in, void* out, int64_t n, float scale, void* stream) {
  return train_cast_scale(in, (act_t*)out, (size_t)n, scale, (cudaStream_t)stream);
}
int vited_train_axpby16(const void* x, float* y, int64_t n, float alpha, float beta, void* stream) {
  return train_act_axpby((const act_t*)x, y, (size_t)n, alpha, beta, (cudaStream_t)stream);
}
int vited_train_axpy32(const float* x, float* y, int64_t n, float alpha, void* stream) {
  return train_f32_axpy(x, y, (size_t)n, alpha, (cudaStream_t)stream);
}
int vited_train_transpose(const void* in, int in_is_f32, int ld_in, void* out, int ld_out, int R, int C, float scale,
                          void* stream) {
  return train_transpose(in, in_is_f32, ld_in, (act_t*)out, ld_out, R, C, scale, (cudaStream_t)stream);
}
int vited_train_ln_forward(const float* x, const float* w, const float* b, void* h, float* stats, int R, int D, float eps,
                           void* stream) {
  return train_ln_forward(x, w, b, (act_t*)h, stats, R, D, eps, (cudaStream_t)stream);
}
int vited_train_ln_backward(const float* dh, const float* x, const float* stats, const float* w, float* dx, float* dw,
                            float* db, int R, int D, float alpha, void* stream) {
  return train_ln_backward(dh, x, stats, w, dx, dw, db, R, D, alpha, (cudaStream_t)stream);
}
int vited_train_gelu_forward(const void* z, void* a, int64_t n, void* stream) {
  return train_gelu_forward((const act_t*)z, (act_t*)a, (size_t)n, (cudaStream_t)stream);
}
int vited_train_gelu_backward(const float* da, const void* z, float* dz, int64_t n, void* stream) {
  return train_gelu_backward(da, (const act_t*)z, dz, (size_t)n, (cudaStream_t)stream);
}
int vited_train_colsum(const float* dy, float* db, int R, int N, float alpha, void* stream) {
  return train_colsum(dy, db, R, N, alpha, (cudaStream_t)stream);
}
int vited_train_gather_rows(const float* in, const int32_t* idx, float* out, int n_blocks, int rows_per, int in_block_stride,
                            int in_row_off, int out_block_stride, int out_row_off, int D, int accumulate, void* stream) {
  return train_gather_rows(in, idx, out, n_blocks, rows_per, in_block_stride, in_row_off, out_block_stride, out_row_off, D,
                           accumulate, (cudaStream_t)stream);
}
int vited_train_scatter_add_rows(const float* src, const int32_t* idx, float* dst, int n_blocks, int rows_per,
                                 int src_block_stride, int src_row_off, int dst_block_stride, int dst_row_off, int D,
                                 float alpha, void* stream) {
  return train_scatter_add_rows(src, idx, dst, n_blocks, rows_per, src_block_stride, src_row_off, dst_block_stride,
                                dst_row_off, D, alpha, (cudaStream_t)stream);
}
int vited_train_attention(int backward, const void* q, int q_ld, const void* k, int k_ld, const void* v, int v_ld, void* o,
                          int o_ld, float* lse, const float* d_o, int do_ld, float* dsum, float* dq, int dq_ld, float* dk,
                          int dk_ld, float* dv, int dv_ld, int n_seq, int H, int hd, int Tq, int Tk, float scale,
                          void* stream) {
  return train_attention(backward, (const act_t*)q, q_ld, (const act_t*)k, k_ld, (const act_t*)v, v_ld, (act_t*)o, o_ld, lse,
                         d_o, do_ld, dsum, dq, dq_ld, dk, dk_ld, dv, dv_ld, n_seq, H, hd, Tq, Tk, scale, (cudaStream_t)stream);
}
int vited_train_bce_logits(const float* logits, const float* labels, int n, float* loss, float* dlogits, float grad_scale,
                           void* stream) {
  return train_bce_logits(logits, labels, n, loss, dlogits, grad_scale, (cudaStream_t)stream);
}
int vited_train_attention_chk(int backward, const void* q, int q_ld, const void* k, int k_ld, const void* v, int v_ld,
                              void* o, int o_ld, float* lse, const float* d_o, int do_ld, float* dsum, float* dq, int dq_ld,
                              float* dk, int dk_ld, float* dv, int dv_ld, int n_seq, int H, int hd, int Tq, int Tk,
                              float scale, int32_t* flag, void* stream) {
  return train_attention(backward, (const act_t*)q, q_ld, (const act_t*)k, k_ld, (const act_t*)v, v_ld, (act_t*)o, o_ld, lse,
                         d_o, do_ld, dsum, dq, dq_ld, dk, dk_ld, dv, dv_ld, n_seq, H, hd, Tq, Tk, scale, (cudaStream_t)stream,
                         flag);
}
float vited_train_range_limit(void) { return train_range_limit(); }
int vited_train_range_check(const void* x, int is_f32, int64_t n, float limit, int32_t* flag, void* stream) {
  return train_range_check(x, is_f32, n, limit, flag, (cudaStream_t)stream);
}
int vited_train_grad_norm(const int64_t* table, int n_tensors, double* partials, int n_partials, float* out_sumsq_and_flag,
                          void* stream) {
  return train_grad_norm(table, n_tensors, partials, n_partials, out_sumsq_and_flag, (cudaStream_t)stream);
}
int vited_train_adamw(const int64_t* table, int n_tensors, int64_t max_numel, double lr, double beta1, double beta2,
                      double eps, float clip_coef, double bias_correction1, double bias_correction2, void* stream) {
  return train_adamw(table, n_tensors, max_numel, lr, beta1, beta2, eps, clip_coef, bias_correction1, bias_correction2,
                     (cudaStream_t)stream);
}

int vited_prepare_pieces(const uint8_t* lab_image, int H, int W, int piece_width, int side, int off, int out_size,
                         float* out, int* n_pieces, void* stream) {
  return prepare_pieces(lab_image, H, W, piece_width, side, off, out_size, out, n_pieces, (cudaStream_t)stream);
}

int vited_normalize_u8(const uint8_t* images, int N, int S, float* out, void* stream) {
  return normalize_u8(images, N, S, out, (cudaStream_t)stream);
}

int vited_retrieval_rows(const float* sim, const int32_t* labels, int N, int32_t* n_relevant, double* ap_sum,
                         int32_t* top1, int32_t* hits10, int32_t* hits100, void* stream) {
  return retrieval_rows(sim, labels, N, n_relevant, ap_sum, top1, hits10, hits100, (cudaStream_t)stream);
}

int vited_puzzle_tables(const float* scores, int flags, const int32_t* order, int N, uint32_t* asym_dist,
                        int64_t* min_dist, int64_t* second_dist, int32_t* n_candidates, int32_t* candidate,
                        float* asym_compat, float* mutual_compat, int32_t* best_buddy, void* stream) {
  return puzzle_tables(scores, flags, order, N, asym_dist, reinterpret_cast<long long*>(min_dist),
                       reinterpret_cast<long long*>(second_dist), n_candidates, candidate, asym_compat, mutual_compat,
                       best_buddy, (cudaStream_t)stream);
}

}  // extern "C"
