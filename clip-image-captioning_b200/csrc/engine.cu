// libclipcap_b200: context, weight ingestion, the three forward stages (ViT -> prefix mapper -> LM) and the
// on-device generation loops behind the C ABI of include/clipcap_b200.h.
//
// Everything here is host orchestration of the kernels in gemm.cu / rowwise.cu / attention.cu / sampler.cu:
// no allocation and no host synchronisation after ccb_create (ccb_generate replays a captured CUDA graph per
// decode step on an internal stream that is fenced against the caller's stream with events).
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "engine.h"

using namespace ccb;

namespace {

thread_local char g_create_err[512] = "";

int fail(ccb_ctx* c, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  if (c)
    c->err = buf;
  else
    snprintf(g_create_err, sizeof(g_create_err), "%s", buf);
  return -1;
}

// run one internal launcher (returns 0 / cudaError / -1 with gemm_last_error) and account for it
#define RUN(call)                                                                                      \
  do {                                                                                                 \
    const int r__ = (call);                                                                            \
    if (r__ != 0) {                                                                                    \
      return fail(c, "%s failed: %s", #call,                                                           \
                  r__ == -1 ? gemm_last_error() : cudaGetErrorString(static_cast<cudaError_t>(r__)));  \
    }                                                                                                  \
    if (c->capturing) c->capture_launches++; else c->launches++;                                       \
  } while (0)

#define CUDA_OK(call)                                                                   \
  do {                                                                                  \
    const cudaError_t e__ = (call);                                                     \
    if (e__ != cudaSuccess) return fail(c, "%s: %s", #call, cudaGetErrorString(e__));   \
  } while (0)

// ------------------------------------------------------------------------------------------ small kernels
__global__ void init_state_kernel(int* block_table, int* block_table_prefill, int max_pages, int rows, int N, int beam,
                                  int S0, int T, int page_tokens, int pages_per_row, int* ctx_len, int* step,
                                  int* lengths, int* stops, uint8_t* finished, float* scores, float* seq_lengths,
                                  uint8_t* has_stopped) {
  const int tid = blockIdx.x * blockDim.x + threadIdx.x;
  const int nth = gridDim.x * blockDim.x;
  if (beam <= 1) {
    // row r owns pages [r * pages_per_row, (r+1) * pages_per_row)
    for (int i = tid; i < rows * pages_per_row; i += nth) {
      const int r = i / pages_per_row, j = i % pages_per_row;
      block_table[static_cast<long long>(r) * max_pages + j] = i;
      block_table_prefill[static_cast<long long>(r) * max_pages + j] = i;
    }
  } else {
    // token-granular pages (page_tokens == 1).  Image n owns pages [n * ppi, (n+1) * ppi), ppi = S0 + beam * T:
    // the first S0 hold the prefix shared by all beams; row k's token written at step j goes to
    // S0 + j * beam + k.  beam_step permutes the entries [0, ctx) of a row, never the fresh ones.
    const int ppi = S0 + beam * T;
    for (int i = tid; i < rows * (S0 + T); i += nth) {
      const int r = i / (S0 + T), j = i % (S0 + T);
      const int n = r / beam, k = r % beam;
      const int page = (j < S0) ? n * ppi + j : n * ppi + S0 + (j - S0) * beam + k;
      block_table[static_cast<long long>(r) * max_pages + j] = page;
      if (k == 0 && j < S0) block_table_prefill[static_cast<long long>(n) * max_pages + j] = page;
    }
  }
  for (int r = tid; r < rows; r += nth) {
    ctx_len[r] = S0;
    lengths[r] = 0;
    stops[r] = 0;
    finished[r] = 0;
    scores[r] = 0.f;
    seq_lengths[r] = 1.f;
    has_stopped[r] = 0;
  }
  if (tid == 0) *step = 0;
}

__global__ void finalize_beam_kernel(const float* scores, const float* seq_lengths, int rows, int* lengths_out,
                                     float* scores_out) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= rows) return;
  const float len = seq_lengths[r];
  if (lengths_out) lengths_out[r] = static_cast<int>(len);
  if (scores_out) scores_out[r] = scores[r] / len;  // inference.py:138
}

// out[n, row_off, :] = wte[token, :]  (BOS embedding appended after the prefix, evaluate_model.py:124-133)
__global__ void token_rows_kernel(const bf16* __restrict__ wte, int token, float* __restrict__ out,
                                  long long image_stride, long long row_off, int d) {
  const bf16* src = wte + static_cast<long long>(token) * d;
  float* dst = out + blockIdx.x * image_stride + row_off * d;
  for (int cidx = threadIdx.x; cidx < d; cidx += blockDim.x) dst[cidx] = __bfloat162float(src[cidx]);
}

// dst[(r / gi) * dgo + r % gi, :] = src[(r / gi) * sgo + soff + r % gi, :]
__global__ void regroup_rows_kernel(const float* __restrict__ src, int gi, int sgo, int soff, float* __restrict__ dst,
                                    int dgo, int d) {
  const int r = blockIdx.x;
  const float4* s4 = reinterpret_cast<const float4*>(src + (static_cast<long long>(r / gi) * sgo + soff + r % gi) * d);
  float4* d4 = reinterpret_cast<float4*>(dst + (static_cast<long long>(r / gi) * dgo + r % gi) * d);
  for (int cidx = threadIdx.x; cidx < d / 4; cidx += blockDim.x) d4[cidx] = s4[cidx];
}

int launch_check() {
  const cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? 0 : static_cast<int>(e);
}

// ------------------------------------------------------------------------------------------ allocation
struct Bump {
  ccb_ctx* c;
  char* cur = nullptr;
  size_t left = 0;
  bool ok = true;
  void* take(size_t bytes) {
    bytes = (bytes + 255) & ~static_cast<size_t>(255);
    if (bytes > left) {
      const size_t chunk = std::max(bytes, static_cast<size_t>(256) << 20);
      void* p = nullptr;
      if (cudaMalloc(&p, chunk) != cudaSuccess) {
        ok = false;
        cudaGetLastError();
        return nullptr;
      }
      c->allocs.push_back(p);
      c->alloc_sizes.push_back(chunk);
      c->device_bytes += static_cast<int64_t>(chunk);
      cur = static_cast<char*>(p);
      left = chunk;
    }
    void* r = cur;
    cur += bytes;
    left -= bytes;
    return r;
  }
  template <typename T>
  T* arr(size_t n) { return static_cast<T*>(take(n * sizeof(T))); }
};

void add_slot(ccb_ctx* c, const std::string& name, WeightSlot::Kind kind, void* dst, long long rows, long long cols,
              long long dst_ld, bool* flag = nullptr, bool optional = false) {
  WeightSlot s;
  s.kind = kind;
  s.dst = dst;
  s.rows = rows;
  s.cols = cols;
  s.dst_ld = dst_ld;
  s.flag = flag;
  s.optional = optional;
  c->slots[name] = s;
}

void make_linear(ccb_ctx* c, Bump& a, Linear& L, int features, int K, bool bias) {
  L.features = features;
  L.K = K;
  L.w = a.arr<bf16>(static_cast<size_t>(features) * K);
  L.bias = a.arr<float>(features);
  L.has_bias = bias;
  (void)c;
}
void make_ln(Bump& a, LayerNormW& n, int d) {
  n.g = a.arr<float>(d);
  n.b = a.arr<float>(d);
}

std::string fmt(const char* f, ...) {
  char buf[256];
  va_list ap;
  va_start(ap, f);
  vsnprintf(buf, sizeof(buf), f, ap);
  va_end(ap);
  return buf;
}

// matrix [features, K] given as nn.Linear [out, in]
void slot_linear(ccb_ctx* c, const std::string& base, Linear& L, bool bias_optional = false) {
  add_slot(c, base + ".weight", WeightSlot::MATRIX, L.w, L.features, L.K, L.ldw ? L.ldw : L.K);
  if (L.has_bias || bias_optional)
    add_slot(c, base + ".bias", WeightSlot::VECTOR_F32, L.bias, L.features, 1, 1, &L.has_bias, bias_optional && !L.has_bias);
}
// HF Conv1D [in, out] -> transposed on ingestion
void slot_conv1d(ccb_ctx* c, const std::string& base, Linear& L) {
  add_slot(c, base + ".weight", WeightSlot::MATRIX_T, L.w, L.K, L.features, L.K);
  add_slot(c, base + ".bias", WeightSlot::VECTOR_F32, L.bias, L.features, 1, 1);
}
void slot_ln(ccb_ctx* c, const std::string& base, LayerNormW& n, int d) {
  add_slot(c, base + ".weight", WeightSlot::VECTOR_F32, n.g, d, 1, 1);
  add_slot(c, base + ".bias", WeightSlot::VECTOR_F32, n.b, d, 1, 1);
}

int act_code(int a) { return a; }  // CCB_ACT_* == ccb::Act

// ------------------------------------------------------------------------------------------ forward pieces
int linear(ccb_ctx* c, const bf16* act, long long lda, int tokens, const Linear& L, int act_fn, const float* residual,
           long long ldr, void* out, long long ldo, int out_bf16, cudaStream_t s) {
  GemmArgs g;
  g.act = act;
  g.lda = lda;
  g.tokens = tokens;
  g.weight = L.w;
  g.ldw = L.ldw;
  g.features = L.features;
  g.K = L.K;
  g.bias = L.has_bias ? L.bias : nullptr;
  g.act_fn = act_fn;
  g.residual = residual;
  g.ldr = ldr;
  g.out = out;
  g.ldo = ldo;
  g.out_bf16 = out_bf16;
  g.allow_pdl = 1;
  return gemm_launch(g, c->gemm_ws, s);
}

struct BlockShape {
  int d, hidden, act;
  float eps;
  bool parallel;  // GPT-J: attn and mlp both read ln_1(h)
};

// one pre-LN block on the residual stream c->h [M, d]; `attn` maps c->qkv [M, 3d] -> c->att [M, d]
template <class AttnFn>
int block_forward(ccb_ctx* c, const Block& b, int M, const BlockShape& sh, AttnFn attn, cudaStream_t s) {
  const int d = sh.d;
  RUN(layernorm_f32_bf16(c->h, d, b.ln1.g, b.ln1.b, sh.eps, c->x, d, M, d, s));
  RUN(linear(c, c->x, d, M, b.qkv, CCB_ACT_NONE, nullptr, 0, c->qkv, 3 * d, 1, s));
  RUN(attn());
  RUN(linear(c, c->att, d, M, b.proj, CCB_ACT_NONE, c->h, d, c->h, d, 0, s));
  if (!sh.parallel) RUN(layernorm_f32_bf16(c->h, d, b.ln2.g, b.ln2.b, sh.eps, c->x, d, M, d, s));
  if (sh.act == CCB_ACT_GEGLU) {
    // fc1 is 2 x hidden wide (layers/Transformer.py:74); the gated product overwrites the first half of every row
    RUN(linear(c, c->x, d, M, b.fc, CCB_ACT_NONE, nullptr, 0, c->mlp, 2 * sh.hidden, 1, s));
    RUN(geglu_inplace(c->mlp, 2 * sh.hidden, M, sh.hidden, s));
    RUN(linear(c, c->mlp, 2 * sh.hidden, M, b.fc2, CCB_ACT_NONE, c->h, d, c->h, d, 0, s));
    return 0;
  }
  RUN(linear(c, c->x, d, M, b.fc, sh.act, nullptr, 0, c->mlp, sh.hidden, 1, s));
  RUN(linear(c, c->mlp, sh.hidden, M, b.fc2, CCB_ACT_NONE, c->h, d, c->h, d, 0, s));
  return 0;
}

// K of the patch-embedding GEMM: 3 * patch^2 rounded up to the GEMM's 64-element K step (patch 14: 588 -> 640)
inline int vit_patch_k(int patch) { return (3 * patch * patch + 63) / 64 * 64; }

int vit_forward(ccb_ctx* c, const void* images, int dtype, int B, float* feat_out, cudaStream_t s, bool all_tokens = false) {
  const ccb_model_desc& D = c->desc;
  if (!D.vit_present) return fail(c, "context was created without an image encoder");
  if (B <= 0 || B > D.max_images) return fail(c, "vit_encode: B=%d outside [1, max_images=%d]", B, D.max_images);
  const int g = D.vit_image / D.vit_patch, np = g * g, w = D.vit_width, S = np + 1, M = B * S;
  const int kpad = vit_patch_k(D.vit_patch);
  RUN(vit_patchify(images, dtype, B, 3, D.vit_image, D.vit_image, D.vit_patch, c->patches, kpad, s));
  RUN(linear(c, c->patches, kpad, B * np, c->vit_conv, CCB_ACT_NONE, nullptr, 0, c->patch_emb, w, 0, s));
  RUN(vit_assemble_lnpre(c->patch_emb, c->vit_cls, c->vit_pos, c->vit_ln_pre.g, c->vit_ln_pre.b, 1e-5f, c->h, B, np, w, s));
  BlockShape sh{w, 4 * w, CCB_ACT_QUICKGELU, 1e-5f, false};
  const int H = D.vit_heads, hd = w / H;
  const float scale = 1.0f / sqrtf(static_cast<float>(hd));
  for (int l = 0; l < D.vit_layers; ++l) {
    auto attn = [&]() {
      return attention_prefill(c->qkv, c->att, B, S, H, hd, scale, 0, nullptr, 0, nullptr, 0, 0, nullptr, s);
    };
    if (block_forward(c, c->vit[l], M, sh, attn, s)) return -1;
  }
  if (all_tokens) {
    // the fork's patched forward (inference.py:421-444): no ln_post, no CLS extraction: x @ proj for every token
    RUN(cast_f32_bf16(c->h, w, c->x, w, M, w, s));
    RUN(linear(c, c->x, w, M, c->vit_proj, CCB_ACT_NONE, nullptr, 0, feat_out, D.vit_out, 0, s));
    return 0;
  }
  // ln_post(x[:, 0, :]) @ proj
  RUN(layernorm_f32_bf16(c->h, static_cast<long long>(S) * w, c->vit_ln_post.g, c->vit_ln_post.b, 1e-5f, c->x, w, B, w, s));
  RUN(linear(c, c->x, w, B, c->vit_proj, CCB_ACT_NONE, nullptr, 0, feat_out, D.vit_out, 0, s));
  return 0;
}

// positions r % ctx and, per sequence, the index of its largest token id (the end-of-text token, OpenAI clip/model.py:
// `x[torch.arange(x.shape[0]), text.argmax(dim=-1)]`; the first maximum wins like torch.argmax)
__global__ void text_positions_eot_kernel(const int* __restrict__ tokens, int ctx, int* __restrict__ positions, int* __restrict__ eot) {
  const int b = blockIdx.x;
  for (int t = threadIdx.x; t < ctx; t += blockDim.x) positions[b * ctx + t] = t;
  if (threadIdx.x == 0) {
    int best = 0, bv = tokens[b * ctx];
    for (int t = 1; t < ctx; ++t) {
      const int v = tokens[b * ctx + t];
      if (v > bv) {
        bv = v;
        best = t;
      }
    }
    eot[b] = best;
  }
}
// dst[b, :] = src[b * ctx + eot[b], :]
__global__ void gather_eot_rows_kernel(const float* __restrict__ src, const int* __restrict__ eot, int ctx, int d, float* __restrict__ dst) {
  const int b = blockIdx.x;
  const float* s = src + (static_cast<long long>(b) * ctx + eot[b]) * d;
  for (int c = threadIdx.x; c < d; c += blockDim.x) dst[static_cast<long long>(b) * d + c] = s[c];
}

// CLIP.encode_text (OpenAI clip/model.py; call sites sampling.py:31, evaluate_model.py ClipScoring): token + positional
// embedding -> causal transformer (QuickGELU) -> ln_final -> row of the end-of-text token @ text_projection
int text_forward(ccb_ctx* c, const int32_t* tokens, int B, float* feat_out, cudaStream_t s) {
  const ccb_model_desc& D = c->desc;
  if (!D.text_present) return fail(c, "context was created without a CLIP text tower");
  if (B <= 0 || B > D.max_texts) return fail(c, "clip_encode_text: B=%d outside [1, max_texts=%d]", B, D.max_texts);
  const int w = D.text_width, S = D.text_ctx, M = B * S, H = D.text_heads, hd = w / H;
  text_positions_eot_kernel<<<B, 128, 0, s>>>(tokens, S, c->txt_positions, c->txt_eot);
  RUN(launch_check());
  RUN(embed_tokens(c->txt_wte, c->txt_wpe, tokens, c->txt_positions, c->h, M, w, D.text_vocab, D.text_ctx, s));
  BlockShape sh{w, 4 * w, CCB_ACT_QUICKGELU, 1e-5f, false};
  const float scale = 1.0f / sqrtf(static_cast<float>(hd));
  for (int l = 0; l < D.text_layers; ++l) {
    auto attn = [&]() {
      return attention_prefill(c->qkv, c->att, B, S, H, hd, scale, 1, nullptr, 0, nullptr, 0, 0, nullptr, s);
    };
    if (block_forward(c, c->txt[l], M, sh, attn, s)) return -1;
  }
  // ln_final is row-wise: gathering the end-of-text rows first is the same arithmetic on B instead of B * ctx rows
  float* rows = reinterpret_cast<float*>(c->mlp);   // [B, w] f32 scratch (the MLP buffer is free here)
  gather_eot_rows_kernel<<<B, 256, 0, s>>>(c->h, c->txt_eot, S, w, rows);
  RUN(launch_check());
  RUN(layernorm_f32_bf16(rows, w, c->txt_ln_final.g, c->txt_ln_final.b, 1e-5f, c->x, w, B, w, s));
  RUN(linear(c, c->x, w, B, c->txt_proj, CCB_ACT_NONE, nullptr, 0, feat_out, D.text_out, 0, s));
  return 0;
}

// feat [B, dim_clip] f32 -> out [B, out_rows_per_image, d] rows [0, P) (out_rows_per_image >= P)
int map_forward(ccb_ctx* c, const float* feat, int B, float* out, int out_rows_per_image, cudaStream_t s) {
  const ccb_model_desc& D = c->desc;
  if (D.map_kind == CCB_MAP_NONE) return fail(c, "context was created without a prefix mapper");
  if (B <= 0 || B > D.max_images) return fail(c, "map_prefix: B=%d outside [1, max_images=%d]", B, D.max_images);
  const int d = D.lm_d, P = D.map_prefix_len, dc = D.map_dim_clip;
  if (D.map_kind != CCB_MAP_TRANSFORMER_ALL) RUN(cast_f32_bf16(feat, dc, c->feat_bf16, dc, B, dc, s));
  if (D.map_kind == CCB_MAP_MLP) {
    // upstream ClipCap MLP mapper: Linear(dc, d*P/2) -> Tanh -> Linear(d*P/2, d*P), viewed as [B, P, d]
    RUN(linear(c, c->feat_bf16, dc, B, c->map_linear, CCB_ACT_TANH, nullptr, 0, c->mlp, D.map_hidden, 1, s));
    RUN(linear(c, c->mlp, D.map_hidden, B, c->map_mlp2, CCB_ACT_NONE, nullptr, 0, out,
               static_cast<long long>(out_rows_per_image) * d, 0, s));
    return 0;
  }
  const int CL = D.map_clip_len, S = CL + P, M = B * S;
  if (D.map_kind == CCB_MAP_TRANSFORMER_ALL) {
    // TransformerMapperAllFeatures.forward (layers/Transformer.py:186-203): feat [B, CL, dc]; x = linear(feat) (+
    // pos_embeddings) per visual token in rows [0, CL) of every sequence, prefix_const in rows [CL, S).  The rows are
    // pre-filled with pos_embeddings (or zeros) and the GEMM adds its result in place (row remap CL -> S).
    RUN(cast_f32_bf16(feat, dc, c->feat_bf16, dc, B * CL, dc, s));
    RUN(mapper_fill_const(c->map_prefix_const, c->h, B, CL, P, d, s));
    RUN(mapper_fill_pos(c->map_pos_present ? c->map_pos : nullptr, c->h, B, CL, P, d, s));
    GemmArgs g;
    g.act = c->feat_bf16;
    g.lda = dc;
    g.tokens = B * CL;
    g.weight = c->map_linear.w;
    g.features = d;
    g.K = dc;
    g.bias = c->map_linear.bias;
    g.residual = c->h;
    g.ldr = d;
    g.out = c->h;
    g.ldo = d;
    g.rg_in = CL;
    g.rg_out = S;
    g.rg_off = 0;
    g.force_orientation = 1;   // the row remap exists only in the normal orientation (the persistent kernels)
    g.allow_pdl = 1;
    RUN(gemm_launch(g, c->gemm_ws, s));
  } else {
  // linear(x).view(B, clip_len, d) lands in rows [0, clip_len) of every sequence (row pitch S*d);
  // rows [clip_len, S) are the learned prefix_const (layers/Transformer.py:154-157)
  RUN(linear(c, c->feat_bf16, dc, B, c->map_linear, CCB_ACT_NONE, nullptr, 0, c->h, static_cast<long long>(S) * d, 0, s));
  RUN(mapper_fill_const(c->map_prefix_const, c->h, B, CL, P, d, s));
  }
  BlockShape sh{d, D.map_hidden, act_code(D.map_act), 1e-5f, false};
  const int H = D.map_heads, hd = d / H;
  const float scale = 1.0f / sqrtf(static_cast<float>(hd));
  for (int l = 0; l < D.map_layers; ++l) {
    auto attn = [&]() {
      return attention_prefill(c->qkv, c->att, B, S, H, hd, scale, 0, nullptr, 0, nullptr, 0, 0, nullptr, s);
    };
    if (block_forward(c, c->mapper[l], M, sh, attn, s)) return -1;
  }
  // out = x[:, clip_len:]  (layers/Transformer.py:159)
  regroup_rows_kernel<<<B * P, 256, 0, s>>>(c->h, P, S, CL, out, out_rows_per_image, d);
  RUN(launch_check());
  return 0;
}

BlockShape lm_shape(const ccb_model_desc& D) {
  return BlockShape{D.lm_d, 4 * D.lm_d, CCB_ACT_GELU_NEW, D.lm_ln_eps, D.lm_arch == CCB_LM_GPTJ};
}

// prefill / teacher-forced pass over embeds [B, S, d]; leaves the final residual stream in c->h
int lm_prefill_layers(ccb_ctx* c, const float* embeds, int B, int S, const uint8_t* key_mask, bool write_cache,
                      cudaStream_t s) {
  const ccb_model_desc& D = c->desc;
  const int d = D.lm_d, M = B * S, H = D.lm_heads, hd = d / H;
  RUN(add_positions(embeds, D.lm_arch == CCB_LM_GPT2 ? c->wpe : nullptr, 0, S, c->h, M, d, s));
  const BlockShape sh = lm_shape(D);
  const float scale = 1.0f / sqrtf(static_cast<float>(hd));
  for (int l = 0; l < D.lm_layers; ++l) {
    auto attn = [&]() {
      return attention_prefill(c->qkv, c->att, B, S, H, hd, scale, 1, write_cache ? &c->kv : nullptr, l,
                               c->block_table_prefill, 0, D.lm_rotary_dim, key_mask, s);
    };
    if (block_forward(c, c->lm[l], M, sh, attn, s)) return -1;
  }
  return 0;
}

// ln_f + lm_head over rows of c->h: all B*S rows, or only the last position of every sequence
int lm_logits(ccb_ctx* c, int B, int S, int last_only, float* logits_out, int64_t ld, cudaStream_t s) {
  const ccb_model_desc& D = c->desc;
  const int d = D.lm_d;
  if (last_only) {
    RUN(layernorm_f32_bf16(c->h + static_cast<long long>(S - 1) * d, static_cast<long long>(S) * d, c->lm_lnf.g,
                           c->lm_lnf.b, D.lm_ln_eps, c->x, d, B, d, s));
    RUN(linear(c, c->x, d, B, c->lm_head, CCB_ACT_NONE, nullptr, 0, logits_out, ld, 0, s));
  } else {
    RUN(layernorm_f32_bf16(c->h, d, c->lm_lnf.g, c->lm_lnf.b, D.lm_ln_eps, c->x, d, B * S, d, s));
    RUN(linear(c, c->x, d, B * S, c->lm_head, CCB_ACT_NONE, nullptr, 0, logits_out, ld, 0, s));
  }
  return 0;
}

// one token per row: embeds next_tokens at position ctx_len, runs all layers against the paged KV cache
bool mega_enabled() {
  static const bool on = [] {
    const char* e = getenv("CCB_MEGA");
    return !(e && e[0] == '0');
  }();
  return on;
}

// the whole layer stack of one decode step as ONE persistent kernel (decode_mega.cu): leaves ln_f(h) in c->x
int lm_decode_layers_mega(ccb_ctx* c, int rows, cudaStream_t s) {
  const ccb_model_desc& D = c->desc;
  const MegaState& m = c->mega;
  MegaParams p;
  memset(&p, 0, sizeof(p));
  p.L = D.lm_layers;
  p.d = D.lm_d;
  p.H = D.lm_heads;
  p.ff = 4 * D.lm_d;
  p.R = rows;
  p.N = (rows + 15) / 16 * 16;
  p.ncta = m.ncta;
  p.eps = D.lm_ln_eps;
  p.scale = 1.0f / sqrtf(static_cast<float>(D.lm_d / D.lm_heads));
  p.layers = m.d_layers;
  p.wmaps = m.d_wmaps;
  p.tile_tbl = m.d_tbl;
  p.tbl_entries = m.tbl_entries;
  for (int k = 0; k < 4; ++k) p.g[k] = m.g[k];
  p.h = c->h;
  p.x = c->x;
  p.att = c->att;
  p.mlp = c->mlp;
  p.ws = m.d_ws;
  p.wte = c->wte;
  p.wpe = c->wpe;
  p.tokens = c->next_tokens;
  p.ctx_len = c->ctx_len;
  p.block_table = c->block_table;
  p.kv = c->kv;
  p.lnf_g = c->lm_lnf.g;
  p.lnf_b = c->lm_lnf.b;
  p.sync = m.d_sync;
  p.sc_cap = (c->max_pages_per_row + 3) & ~3;
  p.trace = m.trace;
  p.log2_page_tokens = 0;
  while ((1 << p.log2_page_tokens) < c->kv.page_tokens) ++p.log2_page_tokens;
  RUN(mega_launch(p, s));
  return 0;
}

int lm_decode_step(ccb_ctx* c, int rows, cudaStream_t s) {
  const ccb_model_desc& D = c->desc;
  const int d = D.lm_d, H = D.lm_heads, hd = d / H;
  if (c->mega.available && rows <= c->mega.max_rows && c->mega.enabled && (c->kv.page_tokens & (c->kv.page_tokens - 1)) == 0) {
    if (lm_decode_layers_mega(c, rows, s)) return -1;
    RUN(linear(c, c->x, d, rows, c->lm_head, CCB_ACT_NONE, nullptr, 0, c->logits, c->ldv, 0, s));
    return 0;
  }
  RUN(embed_tokens(c->wte, D.lm_arch == CCB_LM_GPT2 ? c->wpe : nullptr, c->next_tokens, c->ctx_len, c->h, rows, d, D.lm_vocab, D.lm_n_pos, s));
  const BlockShape sh = lm_shape(D);
  const float scale = 1.0f / sqrtf(static_cast<float>(hd));
  for (int l = 0; l < D.lm_layers; ++l) {
    const Block& b = c->lm[l];
    if (sh.parallel) {
      // GPT-J: h += out_proj(att) + fc_out(gelu_new(fc_in(ln_1 h))) + b as ONE GEMM over K = 5 d.  The 32 x 8 CTAs of the
      // stand-alone out_proj stream 33 MB at 2.6 TB/s (launch ramp, cluster reduce and epilogue around 8 k-blocks per CTA);
      // as the first fifth of fc_out's K loop the same bytes move at that GEMM's 4.9 TB/s.
      const long long ldc = 5LL * d;
      RUN(layernorm_f32_bf16(c->h, d, b.ln1.g, b.ln1.b, sh.eps, c->x, d, rows, d, s));
      RUN(linear(c, c->x, d, rows, b.qkv, CCB_ACT_NONE, nullptr, 0, c->qkv, 3 * d, 1, s));
      RUN(attention_decode(c->qkv, c->attmlp, ldc, rows, H, hd, scale, &c->kv, l, c->block_table, c->ctx_len, D.lm_rotary_dim, s));
      RUN(linear(c, c->x, d, rows, b.fc, sh.act, nullptr, 0, c->attmlp + d, ldc, 1, s));
      RUN(linear(c, c->attmlp, ldc, rows, b.projfc2, CCB_ACT_NONE, c->h, d, c->h, d, 0, s));
      continue;
    }
    auto attn = [&]() {
      return attention_decode(c->qkv, c->att, d, rows, H, hd, scale, &c->kv, l, c->block_table, c->ctx_len,
                              D.lm_rotary_dim, s);
    };
    if (block_forward(c, b, rows, sh, attn, s)) return -1;
  }
  RUN(layernorm_f32_bf16(c->h, d, c->lm_lnf.g, c->lm_lnf.b, D.lm_ln_eps, c->x, d, rows, d, s));
  RUN(linear(c, c->x, d, rows, c->lm_head, CCB_ACT_NONE, nullptr, 0, c->logits, c->ldv, 0, s));
  return 0;
}

SampleParams sample_params(ccb_ctx* c, const ccb_gen_params* p, int rows) {
  SampleParams sp;
  sp.temperature = p->temperature;
  sp.top_p = p->top_p;
  sp.top_k = p->top_k;
  sp.top_p_rows = p->top_p_rows;
  sp.top_k_rows = p->top_k_rows;
  sp.typ_p = p->typ_p;
  sp.typ_p_rows = p->typ_p_rows;
  sp.repetition_penalty = p->repetition_penalty;
  sp.q_noise = p->q_noise;
  sp.ldq = p->q_ld;
  sp.q_step_stride = static_cast<long long>(rows) * p->q_ld;
  sp.seed = p->seed;
  sp.row_ids = reinterpret_cast<const long long*>(p->row_ids);
  (void)c;
  return sp;
}

// token selection for one step of the greedy / sampling loops on c->logits -> c->next_tokens + bookkeeping
int select_step(ccb_ctx* c, const ccb_gen_params* p, int rows, int T, bool after_prefill, cudaStream_t s) {
  const int V = c->desc.lm_vocab;
  if (p->mode == CCB_GEN_GREEDY) {
    RUN(sample_greedy(c->logits, c->ldv, rows, V, c->next_tokens, s));
  } else {
    SampleParams sp = sample_params(c, p, rows);
    sp.history = c->gen_tokens;
    sp.ld_hist = T;
    sp.hist_len_from_step = 1;
    sp.step = c->step;
    RUN(sample_top_p(c->logits, c->ldv, rows, V, sp, c->next_tokens, s));
  }
  RUN(advance_rows(c->next_tokens, rows, c->gen_tokens, T, c->lengths, c->stops, c->finished,
                   after_prefill ? nullptr : c->ctx_len, c->step, p->stop_token, p->max_stops, p->eos_token, s));
  return 0;
}

int beam_select(ccb_ctx* c, const ccb_gen_params* p, int N, int T, bool first, cudaStream_t s) {
  const int beam = p->beam_size, rows = N * beam;
  if (!first) RUN(increment_rows(c->ctx_len, rows, c->step, s));
  BeamState st;
  st.scores = c->scores;
  st.seq_lengths = c->seq_lengths;
  st.has_stopped = c->has_stopped;
  st.tokens = c->gen_tokens;
  st.max_len = T;
  st.step = c->step;
  st.cand_scratch = c->beam_cand;
  st.cand_rows = c->max_rows;
  if (c->capturing) c->capture_launches++; else c->launches++;   // (beam_step launches two kernels)
  RUN(beam_step(c->logits, c->ldv, N, beam, c->desc.lm_vocab, p->temperature, p->stop_token, st, c->next_tokens,
                c->src_rows, c->block_table, c->max_pages_per_row, c->ctx_len, s));
  return 0;
}

int decode_iteration(ccb_ctx* c, const ccb_gen_params* p, int N, int rows, int T, cudaStream_t s) {
  if (lm_decode_step(c, rows, s)) return -1;
  if (p->mode == CCB_GEN_BEAM) return beam_select(c, p, N, T, false, s);
  return select_step(c, p, rows, T, false, s);
}

std::string graph_key(const ccb_gen_params* p, int N, int rows, int T, int c_mega) {
  char buf[512];
  snprintf(buf, sizeof(buf), "g%d m%d N%d r%d T%d st%d ms%d eos%d t%a p%a k%d rp%a b%d seed%llu q%p ld%lld ids%p pr%p kr%p ty%a tr%p",
           c_mega, p->mode, N, rows, T, p->stop_token, p->max_stops, p->eos_token, p->temperature, p->top_p, p->top_k,
           p->repetition_penalty, p->beam_size, static_cast<unsigned long long>(p->seed),
           static_cast<const void*>(p->q_noise), static_cast<long long>(p->q_ld), static_cast<const void*>(p->row_ids),
           static_cast<const void*>(p->top_p_rows), static_cast<const void*>(p->top_k_rows), p->typ_p,
           static_cast<const void*>(p->typ_p_rows));
  return buf;
}

int generate_on_work_stream(ccb_ctx* c, const ccb_gen_params* p, const float* embeds, int N, int S0,
                            int32_t* tokens_out, int32_t* lengths_out, float* scores_out) {
  const ccb_model_desc& D = c->desc;
  cudaStream_t s = c->work;
  const bool is_beam = p->mode == CCB_GEN_BEAM;
  const int beam = is_beam ? p->beam_size : 1;
  const int rows = N * beam;
  const int T = p->max_new_tokens;
  if (p->mode != CCB_GEN_GREEDY && p->mode != CCB_GEN_SAMPLE && !is_beam) return fail(c, "generate: unknown mode %d", p->mode);
  if (N <= 0 || N > D.max_images) return fail(c, "generate: N=%d outside [1, max_images=%d]", N, D.max_images);
  if (beam < 1 || beam > D.max_beam || beam > 8) return fail(c, "generate: beam_size=%d outside [1, max_beam=%d]", beam, D.max_beam);
  if (T <= 0 || S0 <= 0 || S0 + T > D.max_ctx) return fail(c, "generate: S0=%d + max_new_tokens=%d exceeds max_ctx=%d", S0, T, D.max_ctx);
  if (N * S0 > D.max_lm_tokens) return fail(c, "generate: N*S0=%d exceeds max_lm_tokens=%d", N * S0, D.max_lm_tokens);
  if (const char* why = attention_prefill_unsupported(S0, D.lm_d / D.lm_heads, 1, true, D.lm_rotary_dim, false))
    return fail(c, "generate: prefix of S0=%d tokens with head_dim %d: %s", S0, D.lm_d / D.lm_heads, why);

  // KV pool geometry for this call
  const int page_tokens = is_beam ? 1 : D.page_tokens;
  const int pages_per_row = is_beam ? (S0 + T) : (S0 + T + page_tokens - 1) / page_tokens;
  const long long need_tokens = is_beam ? static_cast<long long>(N) * (S0 + static_cast<long long>(beam) * T)
                                        : static_cast<long long>(rows) * pages_per_row * page_tokens;
  if (need_tokens > c->kv_pool_tokens) return fail(c, "generate: KV pool too small (%lld > %lld tokens)", need_tokens, c->kv_pool_tokens);
  c->kv.page_tokens = page_tokens;
  c->kv.num_pages = static_cast<int>(c->kv_pool_tokens / page_tokens);
  c->kv.max_pages_per_row = c->max_pages_per_row;

  init_state_kernel<<<148, 256, 0, s>>>(c->block_table, c->block_table_prefill, c->max_pages_per_row, rows, N, beam, S0,
                                        T, page_tokens, pages_per_row, c->ctx_len, c->step, c->lengths, c->stops,
                                        c->finished, c->scores, c->seq_lengths, c->has_stopped);
  RUN(launch_check());
  CUDA_OK(cudaMemsetAsync(c->gen_tokens, 0, sizeof(int) * static_cast<size_t>(rows) * T, s));

  const int slot = static_cast<int>(c->generate_calls % ccb_ctx::kTimingSlots);
  CUDA_OK(cudaEventRecord(c->ev_t0[slot], s));
  // ---- prefill: one pass over the prefix, K/V written to the cache, logits of the last position
  if (lm_prefill_layers(c, embeds, N, S0, nullptr, true, s)) return -1;
  if (lm_logits(c, N, S0, 1, c->logits, c->ldv, s)) return -1;
  if (is_beam) {
    if (beam_select(c, p, N, T, true, s)) return -1;
  } else {
    if (select_step(c, p, rows, T, true, s)) return -1;
  }
  CUDA_OK(cudaEventRecord(c->ev_t1[slot], s));

  // ---- decode: T-1 replays of one captured step (every kernel reads step / ctx_len from device memory)
  if (T > 1) {
    const std::string key = graph_key(p, N, rows, T, c->mega.enabled ? 1 : 0);
    auto it = c->graphs.find(key);
    if (it == c->graphs.end()) {
      cudaGraph_t graph = nullptr;
      CUDA_OK(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
      c->capturing = true;
      c->capture_launches = 0;
      const int r = decode_iteration(c, p, N, rows, T, s);
      c->capturing = false;
      const cudaError_t e = cudaStreamEndCapture(s, &graph);
      if (r != 0) {
        if (graph) cudaGraphDestroy(graph);
        return -1;
      }
      if (e != cudaSuccess) return fail(c, "cudaStreamEndCapture: %s", cudaGetErrorString(e));
      GraphEntry ge;
      ge.nodes = c->capture_launches;
      const cudaError_t e2 = cudaGraphInstantiate(&ge.exec, graph, 0);
      cudaGraphDestroy(graph);
      if (e2 != cudaSuccess) return fail(c, "cudaGraphInstantiate: %s", cudaGetErrorString(e2));
      if (c->graphs.size() >= 32) {  // bound the cache
        for (auto& kvp : c->graphs) cudaGraphExecDestroy(kvp.second.exec);
        c->graphs.clear();
      }
      it = c->graphs.emplace(key, ge).first;
    }
    for (int t = 1; t < T; ++t) {
      CUDA_OK(cudaGraphLaunch(it->second.exec, s));
      c->launches += it->second.nodes;
    }
  }
  CUDA_OK(cudaEventRecord(c->ev_t2[slot], s));
  c->timing_steps[slot] = T - 1;
  c->generate_calls++;

  // ---- results
  CUDA_OK(cudaMemcpyAsync(tokens_out, c->gen_tokens, sizeof(int) * static_cast<size_t>(rows) * T, cudaMemcpyDeviceToDevice, s));
  if (is_beam) {
    finalize_beam_kernel<<<(rows + 255) / 256, 256, 0, s>>>(c->scores, c->seq_lengths, rows, lengths_out, scores_out);
    RUN(launch_check());
  } else if (lengths_out) {
    CUDA_OK(cudaMemcpyAsync(lengths_out, c->lengths, sizeof(int) * rows, cudaMemcpyDeviceToDevice, s));
  }
  return 0;
}

int fence_in(ccb_ctx* c, cudaStream_t caller) {
  CUDA_OK(cudaEventRecord(c->ev_in, caller));
  CUDA_OK(cudaStreamWaitEvent(c->work, c->ev_in, 0));
  return 0;
}
int fence_out(ccb_ctx* c, cudaStream_t caller) {
  CUDA_OK(cudaEventRecord(c->ev_out, c->work));
  CUDA_OK(cudaStreamWaitEvent(caller, c->ev_out, 0));
  return 0;
}

bool starts_with(const char* s, const char* prefix, const char** rest) {
  const size_t n = strlen(prefix);
  if (strncmp(s, prefix, n) == 0) {
    *rest = s + n;
    return true;
  }
  return false;
}

}  // namespace

// ================================================================================================ C ABI
extern "C" {

// Every entry point runs with the context's device current (launches, function attributes and event calls are per device)
// and restores the caller's device on the way out.
struct DeviceGuard {
  int prev = -1, dev;
  explicit DeviceGuard(int d) : dev(d) {
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    if (prev != dev) cudaSetDevice(dev);
  }
  ~DeviceGuard() {
    if (prev >= 0 && prev != dev) cudaSetDevice(prev);
  }
};

const char* ccb_last_error(const ccb_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_err; }

int64_t ccb_device_bytes(const ccb_ctx* ctx) { return ctx ? ctx->device_bytes : 0; }
int64_t ccb_launch_count(const ccb_ctx* ctx) { return ctx ? ctx->launches : 0; }

void ccb_destroy(ccb_ctx* c) {
  if (!c) return;
  DeviceGuard dev_guard(c->device);
  cudaDeviceSynchronize();
  for (auto& kvp : c->graphs) cudaGraphExecDestroy(kvp.second.exec);
  for (void* p : c->allocs) cudaFree(p);
  if (c->work) cudaStreamDestroy(c->work);
  for (cudaEvent_t e : {c->ev_in, c->ev_out})
    if (e) cudaEventDestroy(e);
  for (int i = 0; i < ccb_ctx::kTimingSlots; ++i)
    for (cudaEvent_t e : {c->ev_t0[i], c->ev_t1[i], c->ev_t2[i]})
      if (e) cudaEventDestroy(e);
  delete c;
}

int ccb_create(ccb_ctx** out, const ccb_model_desc* desc, int device) {
  if (!out || !desc) return fail(nullptr, "ccb_create: null argument");
  *out = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    return fail(nullptr, "ccb_create: no CUDA device (this library has no CPU fallback)");
  }
  if (device < 0 || device >= ndev) return fail(nullptr, "ccb_create: device %d out of range (%d devices)", device, ndev);
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return fail(nullptr, "ccb_create: cudaGetDeviceProperties failed");
  if (prop.major != 10) return fail(nullptr, "ccb_create: device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor);
  DeviceGuard dev_guard(device);   // (the caller's current device is restored on return)
  {
    int cur = -1;
    if (cudaGetDevice(&cur) != cudaSuccess || cur != device) return fail(nullptr, "ccb_create: cudaSetDevice failed");
  }

  const ccb_model_desc& D = *desc;
  if (D.lm_d <= 0 || D.lm_layers <= 0 || D.lm_heads <= 0 || D.lm_vocab <= 0 || D.lm_d % D.lm_heads)
    return fail(nullptr, "ccb_create: bad language-model dimensions");
  if (D.lm_d % 64) return fail(nullptr, "ccb_create: lm_d must be a multiple of 64");
  const int lm_hd = D.lm_d / D.lm_heads;
  if (lm_hd != 64 && lm_hd != 128 && lm_hd != 256) return fail(nullptr, "ccb_create: LM head_dim %d unsupported (64/128/256)", lm_hd);
  if (D.lm_arch != CCB_LM_GPT2 && D.lm_arch != CCB_LM_GPTJ) return fail(nullptr, "ccb_create: unknown lm_arch");
  if (D.lm_arch == CCB_LM_GPT2 && D.max_ctx > D.lm_n_pos)
    return fail(nullptr, "ccb_create: max_ctx=%d exceeds the model's %d learned positions (wpe)", D.max_ctx, D.lm_n_pos);
  if (D.max_images <= 0 || D.max_beam <= 0 || D.max_ctx <= 0 || D.max_lm_tokens <= 0 || D.page_tokens <= 0)
    return fail(nullptr, "ccb_create: capacities must be positive");
  if ((D.map_kind == CCB_MAP_TRANSFORMER || D.map_kind == CCB_MAP_TRANSFORMER_ALL) && (D.map_heads <= 0 || D.lm_d % D.map_heads || (D.lm_d / D.map_heads) % 2 ||
                                            D.map_hidden % 64 || D.map_dim_clip % 64))
    return fail(nullptr, "ccb_create: bad mapper dimensions");
  if (D.map_kind == CCB_MAP_MLP && (D.map_hidden % 64 || D.map_dim_clip % 64)) return fail(nullptr, "ccb_create: bad MLP mapper dimensions");
  // any patch size that divides the image (patch 14: the K of the patch GEMM is padded, see vit_patch_k)
  if (D.vit_present && (D.vit_width % 64 || D.vit_heads <= 0 || D.vit_width % D.vit_heads || D.vit_patch <= 0 || D.vit_image % D.vit_patch))
    return fail(nullptr, "ccb_create: bad ViT dimensions");
  if (D.text_present && (D.text_width % 64 || D.text_heads <= 0 || D.text_width % D.text_heads || (D.text_width / D.text_heads) % 16 ||
                         D.text_ctx <= 0 || D.text_ctx > 128 || D.text_vocab <= 0 || D.text_out <= 0 || D.max_texts <= 0))
    return fail(nullptr, "ccb_create: bad CLIP text-tower dimensions");
  // every fixed-length attention of the context must have a kernel (the LM's prefill length is checked per call)
  {
    struct { bool present; const char* what; int S, hd, causal; } att[] = {
        {D.vit_present != 0, "ViT", D.vit_present ? (D.vit_image / D.vit_patch) * (D.vit_image / D.vit_patch) + 1 : 0,
         D.vit_present ? D.vit_width / D.vit_heads : 0, 0},
        {D.text_present != 0, "CLIP text tower", D.text_ctx, D.text_present ? D.text_width / D.text_heads : 0, 1},
        {D.map_kind == CCB_MAP_TRANSFORMER || D.map_kind == CCB_MAP_TRANSFORMER_ALL, "mapper", D.map_clip_len + D.map_prefix_len,
         D.map_heads > 0 ? D.lm_d / D.map_heads : 0, 0}};
    for (const auto& a : att) {
      const char* why = a.present ? attention_prefill_unsupported(a.S, a.hd, a.causal, false, 0, false) : nullptr;
      if (why) return fail(nullptr, "ccb_create: %s attention over %d tokens with head_dim %d: %s", a.what, a.S, a.hd, why);
    }
  }

  ccb_ctx* c = new ccb_ctx();
  c->desc = D;
  c->device = device;
  c->num_sms = prop.multiProcessorCount;
  if (gemm_init(device) != 0) {
    fail(nullptr, "ccb_create: %s", gemm_last_error());
    delete c;
    return -1;
  }
  Bump a{c};
  const int d = D.lm_d, V = D.lm_vocab;

  // ---- language model
  c->wte = a.arr<bf16>(static_cast<size_t>(V) * d);
  add_slot(c, "transformer.wte.weight", WeightSlot::ROWS_BF16, c->wte, V, d, d);
  if (D.lm_arch == CCB_LM_GPT2) {
    c->wpe = a.arr<bf16>(static_cast<size_t>(D.lm_n_pos) * d);
    add_slot(c, "transformer.wpe.weight", WeightSlot::ROWS_BF16, c->wpe, D.lm_n_pos, d, d);
  }
  c->lm.resize(D.lm_layers);
  for (int l = 0; l < D.lm_layers; ++l) {
    Block& b = c->lm[l];
    const std::string base = fmt("transformer.h.%d", l);
    make_ln(a, b.ln1, d);
    slot_ln(c, base + ".ln_1", b.ln1, d);
    if (D.lm_arch == CCB_LM_GPT2) {
      make_ln(a, b.ln2, d);
      slot_ln(c, base + ".ln_2", b.ln2, d);
      make_linear(c, a, b.qkv, 3 * d, d, true);
      make_linear(c, a, b.proj, d, d, true);
      make_linear(c, a, b.fc, 4 * d, d, true);
      make_linear(c, a, b.fc2, d, 4 * d, true);
      slot_conv1d(c, base + ".attn.c_attn", b.qkv);
      slot_conv1d(c, base + ".attn.c_proj", b.proj);
      slot_conv1d(c, base + ".mlp.c_fc", b.fc);
      slot_conv1d(c, base + ".mlp.c_proj", b.fc2);
    } else {
      make_linear(c, a, b.qkv, 3 * d, d, false);
      make_linear(c, a, b.fc, 4 * d, d, true);
      {
        // out_proj | fc_out side by side in one [d, 5d] matrix (engine.h: Block::projfc2); the prefill GEMMs read the two
        // column ranges through their row pitch
        bf16* cat = a.arr<bf16>(static_cast<size_t>(d) * 5 * d);
        b.proj.w = cat;
        b.proj.features = d;
        b.proj.K = d;
        b.proj.ldw = 5LL * d;
        b.proj.bias = a.arr<float>(d);
        b.proj.has_bias = false;
        b.fc2.w = cat + d;
        b.fc2.features = d;
        b.fc2.K = 4 * d;
        b.fc2.ldw = 5LL * d;
        b.fc2.bias = a.arr<float>(d);
        b.fc2.has_bias = true;
        b.projfc2 = b.fc2;
        b.projfc2.w = cat;
        b.projfc2.K = 5 * d;
      }
      add_slot(c, base + ".attn.q_proj.weight", WeightSlot::MATRIX, b.qkv.w, d, d, d);
      add_slot(c, base + ".attn.k_proj.weight", WeightSlot::MATRIX, b.qkv.w + static_cast<size_t>(d) * d, d, d, d);
      add_slot(c, base + ".attn.v_proj.weight", WeightSlot::MATRIX, b.qkv.w + 2 * static_cast<size_t>(d) * d, d, d, d);
      slot_linear(c, base + ".attn.out_proj", b.proj);
      slot_linear(c, base + ".mlp.fc_in", b.fc);
      slot_linear(c, base + ".mlp.fc_out", b.fc2);
    }
  }
  make_ln(a, c->lm_lnf, d);
  slot_ln(c, "transformer.ln_f", c->lm_lnf, d);
  if (D.lm_arch == CCB_LM_GPT2) {
    c->lm_head.w = c->wte;  // tied
    c->lm_head.features = V;
    c->lm_head.K = d;
    c->lm_head.has_bias = false;
  } else {
    make_linear(c, a, c->lm_head, V, d, true);
    slot_linear(c, "lm_head", c->lm_head);
  }

  // ---- mapper
  int map_S = 0;
  if (D.map_kind == CCB_MAP_TRANSFORMER || D.map_kind == CCB_MAP_TRANSFORMER_ALL) {
    map_S = D.map_clip_len + D.map_prefix_len;
    if (D.map_kind == CCB_MAP_TRANSFORMER_ALL) {
      make_linear(c, a, c->map_linear, d, D.map_dim_clip, true);
      c->map_pos = a.arr<float>(static_cast<size_t>(D.map_clip_len) * d);
      add_slot(c, "clip_project.pos_embeddings", WeightSlot::VECTOR_F32, c->map_pos, static_cast<long long>(D.map_clip_len) * d,
               1, 1, &c->map_pos_present, true);   // optional (use_pos_embeddings, layers/Transformer.py:181-185)
    } else {
      make_linear(c, a, c->map_linear, D.map_clip_len * d, D.map_dim_clip, true);
    }
    slot_linear(c, "clip_project.linear", c->map_linear);
    c->map_prefix_const = a.arr<float>(static_cast<size_t>(D.map_prefix_len) * d);
    add_slot(c, "clip_project.prefix_const", WeightSlot::VECTOR_F32, c->map_prefix_const,
             static_cast<long long>(D.map_prefix_len) * d, 1, 1);
    c->mapper.resize(D.map_layers);
    for (int l = 0; l < D.map_layers; ++l) {
      Block& b = c->mapper[l];
      const std::string base = fmt("clip_project.transformer.layers.%d", l);
      make_ln(a, b.ln1, d);
      make_ln(a, b.ln2, d);
      slot_ln(c, base + ".norm1", b.ln1, d);
      slot_ln(c, base + ".norm2", b.ln2, d);
      make_linear(c, a, b.qkv, 3 * d, d, false);
      make_linear(c, a, b.proj, d, d, true);
      make_linear(c, a, b.fc, (D.map_act == CCB_ACT_GEGLU ? 2 : 1) * D.map_hidden, d, true);
      make_linear(c, a, b.fc2, d, D.map_hidden, true);
      // to_queries [d, d] -> rows [0, d); to_keys_values [2d, d] -> rows [d, 3d): keys then values
      // (layers/MultiHeadAttention.py:24-30).  The projections are bias-free by default (Transformer.py:91,96).
      add_slot(c, base + ".attn.to_queries.weight", WeightSlot::MATRIX, b.qkv.w, d, d, d);
      add_slot(c, base + ".attn.to_keys_values.weight", WeightSlot::MATRIX, b.qkv.w + static_cast<size_t>(d) * d, 2 * d, d, d);
      add_slot(c, base + ".attn.to_queries.bias", WeightSlot::VECTOR_F32, b.qkv.bias, d, 1, 1, &b.qkv.has_bias, true);
      add_slot(c, base + ".attn.to_keys_values.bias", WeightSlot::VECTOR_F32, b.qkv.bias + d, 2 * d, 1, 1, &b.qkv.has_bias, true);
      slot_linear(c, base + ".attn.project", b.proj);
      slot_linear(c, base + ".mlp.fc1", b.fc);
      slot_linear(c, base + ".mlp.fc2", b.fc2);
    }
  } else if (D.map_kind == CCB_MAP_MLP) {
    make_linear(c, a, c->map_linear, D.map_hidden, D.map_dim_clip, true);
    make_linear(c, a, c->map_mlp2, D.map_prefix_len * d, D.map_hidden, true);
    slot_linear(c, "clip_project.model.0", c->map_linear);
    slot_linear(c, "clip_project.model.2", c->map_mlp2);
  }

  // ---- ViT
  int vit_S = 0;
  if (D.vit_present) {
    const int w = D.vit_width, g = D.vit_image / D.vit_patch, np = g * g, kdim = 3 * D.vit_patch * D.vit_patch;
    vit_S = np + 1;
    // conv1 as a [w, kdim] matrix at the padded pitch of the patch rows; the pad columns stay zero (the arena is cleared)
    make_linear(c, a, c->vit_conv, w, vit_patch_k(D.vit_patch), false);
    add_slot(c, "visual.conv1.weight", WeightSlot::MATRIX, c->vit_conv.w, w, kdim, vit_patch_k(D.vit_patch));
    c->vit_cls = a.arr<float>(w);
    c->vit_pos = a.arr<float>(static_cast<size_t>(vit_S) * w);
    add_slot(c, "visual.class_embedding", WeightSlot::VECTOR_F32, c->vit_cls, w, 1, 1);
    add_slot(c, "visual.positional_embedding", WeightSlot::VECTOR_F32, c->vit_pos, static_cast<long long>(vit_S) * w, 1, 1);
    make_ln(a, c->vit_ln_pre, w);
    make_ln(a, c->vit_ln_post, w);
    slot_ln(c, "visual.ln_pre", c->vit_ln_pre, w);
    slot_ln(c, "visual.ln_post", c->vit_ln_post, w);
    c->vit.resize(D.vit_layers);
    for (int l = 0; l < D.vit_layers; ++l) {
      Block& b = c->vit[l];
      const std::string base = fmt("visual.transformer.resblocks.%d", l);
      make_ln(a, b.ln1, w);
      make_ln(a, b.ln2, w);
      slot_ln(c, base + ".ln_1", b.ln1, w);
      slot_ln(c, base + ".ln_2", b.ln2, w);
      make_linear(c, a, b.qkv, 3 * w, w, true);
      make_linear(c, a, b.proj, w, w, true);
      make_linear(c, a, b.fc, 4 * w, w, true);
      make_linear(c, a, b.fc2, w, 4 * w, true);
      add_slot(c, base + ".attn.in_proj_weight", WeightSlot::MATRIX, b.qkv.w, 3 * w, w, w);
      add_slot(c, base + ".attn.in_proj_bias", WeightSlot::VECTOR_F32, b.qkv.bias, 3 * w, 1, 1);
      slot_linear(c, base + ".attn.out_proj", b.proj);
      slot_linear(c, base + ".mlp.c_fc", b.fc);
      slot_linear(c, base + ".mlp.c_proj", b.fc2);
    }
    make_linear(c, a, c->vit_proj, D.vit_out, w, false);
    add_slot(c, "visual.proj", WeightSlot::MATRIX_T, c->vit_proj.w, w, D.vit_out, w);  // proj [w, out] -> [out, w]
  }

  // ---- CLIP text tower (OpenAI names under "clip_text.": token_embedding.weight, positional_embedding,
  //      transformer.resblocks.N.*, ln_final.*, text_projection)
  if (D.text_present) {
    const int w = D.text_width;
    c->txt_wte = a.arr<bf16>(static_cast<size_t>(D.text_vocab) * w);
    c->txt_wpe = a.arr<bf16>(static_cast<size_t>(D.text_ctx) * w);
    add_slot(c, "clip_text.token_embedding.weight", WeightSlot::ROWS_BF16, c->txt_wte, D.text_vocab, w, w);
    add_slot(c, "clip_text.positional_embedding", WeightSlot::ROWS_BF16, c->txt_wpe, D.text_ctx, w, w);
    make_ln(a, c->txt_ln_final, w);
    slot_ln(c, "clip_text.ln_final", c->txt_ln_final, w);
    c->txt.resize(D.text_layers);
    for (int l = 0; l < D.text_layers; ++l) {
      Block& b = c->txt[l];
      const std::string base = fmt("clip_text.transformer.resblocks.%d", l);
      make_ln(a, b.ln1, w);
      make_ln(a, b.ln2, w);
      slot_ln(c, base + ".ln_1", b.ln1, w);
      slot_ln(c, base + ".ln_2", b.ln2, w);
      make_linear(c, a, b.qkv, 3 * w, w, true);
      make_linear(c, a, b.proj, w, w, true);
      make_linear(c, a, b.fc, 4 * w, w, true);
      make_linear(c, a, b.fc2, w, 4 * w, true);
      add_slot(c, base + ".attn.in_proj_weight", WeightSlot::MATRIX, b.qkv.w, 3 * w, w, w);
      add_slot(c, base + ".attn.in_proj_bias", WeightSlot::VECTOR_F32, b.qkv.bias, 3 * w, 1, 1);
      slot_linear(c, base + ".attn.out_proj", b.proj);
      slot_linear(c, base + ".mlp.c_fc", b.fc);
      slot_linear(c, base + ".mlp.c_proj", b.fc2);
    }
    make_linear(c, a, c->txt_proj, D.text_out, w, false);
    add_slot(c, "clip_text.text_projection", WeightSlot::MATRIX_T, c->txt_proj.w, w, D.text_out, w);  // [w, out] -> [out, w]
    c->txt_positions = a.arr<int>(static_cast<size_t>(D.max_texts) * D.text_ctx);
    c->txt_eot = a.arr<int>(D.max_texts);
  }

  // ---- workspaces
  c->max_rows = D.max_images * D.max_beam;
  int M = std::max(D.max_lm_tokens, c->max_rows);
  M = std::max(M, D.max_images * map_S);
  M = std::max(M, D.max_images * vit_S);
  if (D.text_present) M = std::max(M, D.max_texts * D.text_ctx);
  c->max_rows_tokens = M;
  c->dmax = std::max(d, std::max(D.vit_present ? D.vit_width : 0, D.text_present ? D.text_width : 0));
  c->hidden_max = std::max(4 * d, std::max(D.map_kind != CCB_MAP_NONE ? (D.map_act == CCB_ACT_GEGLU ? 2 : 1) * D.map_hidden : 0,
                                           D.vit_present ? 4 * D.vit_width : 0));
  if (D.text_present) c->hidden_max = std::max(c->hidden_max, 4 * D.text_width);
  const size_t Mz = static_cast<size_t>(M);
  c->h = a.arr<float>(Mz * c->dmax);
  c->x = a.arr<bf16>(Mz * c->dmax);
  c->qkv = a.arr<bf16>(Mz * 3 * c->dmax);
  c->att = a.arr<bf16>(Mz * c->dmax);
  c->mlp = a.arr<bf16>(Mz * c->hidden_max);
  if (D.lm_arch == CCB_LM_GPTJ) c->attmlp = a.arr<bf16>(static_cast<size_t>(c->max_rows) * 5 * d);
  if (D.vit_present) {
    const int g = D.vit_image / D.vit_patch, np = g * g;
    c->patches = a.arr<bf16>(static_cast<size_t>(D.max_images) * np * vit_patch_k(D.vit_patch));
    c->patch_emb = a.arr<float>(static_cast<size_t>(D.max_images) * np * D.vit_width);
  }
  const int dc = std::max(D.map_dim_clip, D.vit_present ? D.vit_out : 0);
  const int feat_tokens = D.map_kind == CCB_MAP_TRANSFORMER_ALL ? std::max(D.map_clip_len, vit_S) : 1;   // per image
  c->feat = a.arr<float>(static_cast<size_t>(D.max_images) * feat_tokens * std::max(dc, 1));
  c->feat_bf16 = a.arr<bf16>(static_cast<size_t>(D.max_images) * feat_tokens * std::max(dc, 1));
  c->prefix = a.arr<float>(static_cast<size_t>(D.max_images) * (std::max(D.map_prefix_len, 0) + 1) * d);
  c->ldv = (static_cast<int64_t>(V) + 63) / 64 * 64;
  c->logits = a.arr<float>(static_cast<size_t>(std::max(c->max_rows, D.max_images)) * c->ldv);
  c->gemm_ws.ws_bytes = static_cast<size_t>(96) << 20;
  c->gemm_ws.ws = static_cast<float*>(a.take(c->gemm_ws.ws_bytes));
  c->gemm_ws.sem_count = 8192;
  c->gemm_ws.sem = a.arr<int>(c->gemm_ws.sem_count);
  c->gemm_ws.num_sms = c->num_sms;

  // ---- KV pool + state
  const int lm_H = D.lm_heads;
  c->kv.L = D.lm_layers;
  c->kv.H = lm_H;
  c->kv.hd = lm_hd;
  const long long ctx_round = (static_cast<long long>(D.max_ctx) + D.page_tokens - 1) / D.page_tokens * D.page_tokens;
  c->kv_pool_tokens = static_cast<long long>(c->max_rows) * ctx_round;
  c->kv.base = a.arr<bf16>(static_cast<size_t>(2) * D.lm_layers * c->kv_pool_tokens * d);
  c->max_pages_per_row = D.max_ctx;
  c->block_table = a.arr<int>(static_cast<size_t>(c->max_rows) * c->max_pages_per_row);
  c->block_table_prefill = a.arr<int>(static_cast<size_t>(D.max_images) * c->max_pages_per_row);
  c->ctx_len = a.arr<int>(c->max_rows);
  c->step = a.arr<int>(1);
  c->next_tokens = a.arr<int>(c->max_rows);
  c->src_rows = a.arr<int>(c->max_rows);
  c->beam_cand = a.take(static_cast<size_t>(c->max_rows) * kBeamCandPerRow * 8);
  c->gen_tokens = a.arr<int>(static_cast<size_t>(c->max_rows) * D.max_ctx);
  c->lengths = a.arr<int>(c->max_rows);
  c->stops = a.arr<int>(c->max_rows);
  c->finished = a.arr<uint8_t>(c->max_rows);
  c->scores = a.arr<float>(c->max_rows);
  c->seq_lengths = a.arr<float>(c->max_rows);
  c->has_stopped = a.arr<uint8_t>(c->max_rows);
  c->bos_token = a.arr<int>(D.max_images);

  // ---- persistent decode kernel: GPT-2 blocks with head_dim 64 (every GPT-2 size), up to 256 rows per step
  MegaState& mg = c->mega;
  if (D.lm_arch == CCB_LM_GPT2 && lm_hd == 64 && d <= 4096 && mega_init() == 0) {
    mega_plan(mg, d, 4 * d, c->num_sms);
    if (mg.tbl_entries <= 256) {
      mg.max_rows = std::min(c->max_rows, 256);
      mg.d_wmaps = static_cast<CUtensorMap*>(a.take(sizeof(CUtensorMap) * 4 * D.lm_layers));
      mg.d_layers = a.arr<MegaLayer>(D.lm_layers);
      mg.d_tbl = a.arr<uint32_t>(mg.tbl_entries);
      mg.d_ws = a.arr<float>(mg.ws_floats_per_row * mg.max_rows);
      mg.d_sync = a.arr<unsigned int>(64);
      mg.available = true;
      mg.enabled = mega_enabled();
    }
  }

  if (!a.ok) {
    fail(nullptr, "ccb_create: out of device memory after %lld bytes", static_cast<long long>(c->device_bytes));
    ccb_destroy(c);
    return -1;
  }
  // zero everything once (optional biases, semaphores, block tables)
  for (size_t i = 0; i < c->allocs.size(); ++i) cudaMemset(c->allocs[i], 0, c->alloc_sizes[i]);
  if (mg.available) {
    // weight tensor maps (addresses are fixed from here on; the values arrive through ccb_load_weight)
    std::vector<CUtensorMap> maps(static_cast<size_t>(4) * D.lm_layers);
    std::vector<MegaLayer> lys(D.lm_layers);
    bool ok = true;
    for (int l = 0; l < D.lm_layers && ok; ++l) {
      const Block& b = c->lm[l];
      const Linear* lin[4] = {&b.qkv, &b.proj, &b.fc, &b.fc2};
      for (int k = 0; k < 4; ++k)
        ok = ok && gemm_make_tmap(&maps[l * 4 + k], lin[k]->w, lin[k]->features, lin[k]->K, lin[k]->K, 128) == 0;
      lys[l] = MegaLayer{b.ln1.g, b.ln1.b, b.ln2.g, b.ln2.b, b.qkv.bias, b.proj.bias, b.fc.bias, b.fc2.bias};
    }
    ok = ok && cudaMemcpy(mg.d_wmaps, maps.data(), maps.size() * sizeof(CUtensorMap), cudaMemcpyHostToDevice) == cudaSuccess;
    ok = ok && cudaMemcpy(mg.d_layers, lys.data(), lys.size() * sizeof(MegaLayer), cudaMemcpyHostToDevice) == cudaSuccess;
    ok = ok && cudaMemcpy(mg.d_tbl, mg.h_tbl.data(), mg.h_tbl.size() * sizeof(uint32_t), cudaMemcpyHostToDevice) == cudaSuccess;
    if (!ok) {
      fail(nullptr, "ccb_create: persistent decode kernel setup failed: %s", gemm_last_error());
      ccb_destroy(c);
      return -1;
    }
  }
  if (cudaStreamCreateWithFlags(&c->work, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&c->ev_in, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&c->ev_out, cudaEventDisableTiming) != cudaSuccess ||
      cudaDeviceSynchronize() != cudaSuccess) {
    fail(nullptr, "ccb_create: stream / event creation failed: %s", cudaGetErrorString(cudaGetLastError()));
    ccb_destroy(c);
    return -1;
  }
  for (int i = 0; i < ccb_ctx::kTimingSlots; ++i) {
    if (cudaEventCreate(&c->ev_t0[i]) != cudaSuccess || cudaEventCreate(&c->ev_t1[i]) != cudaSuccess ||
        cudaEventCreate(&c->ev_t2[i]) != cudaSuccess) {
      fail(nullptr, "ccb_create: event creation failed");
      ccb_destroy(c);
      return -1;
    }
  }
  *out = c;
  return 0;
}

int ccb_load_weight(ccb_ctx* c, const char* name, const void* dev_ptr, int dtype, const int64_t* shape, int ndim,
                    void* stream) {
  if (!c || !name || !dev_ptr || !shape) return fail(c, "ccb_load_weight: null argument");
  DeviceGuard dev_guard(c->device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  // normalise the reference's module prefixes (SURVEY appendix B.3)
  std::string key;
  const char* rest = nullptr;
  if (starts_with(name, "language_model.", &rest)) key = rest;
  else if (starts_with(name, "visual_encoder.", &rest)) key = std::string("visual.") + rest;
  else key = name;
  auto it = c->slots.find(key);
  if (it == c->slots.end()) return 1;  // not used by this context
  WeightSlot& w = it->second;
  long long numel = 1;
  for (int i = 0; i < ndim; ++i) numel *= shape[i];
  if (numel != w.rows * w.cols) return fail(c, "ccb_load_weight(%s): expected %lld elements, got %lld", name, w.rows * w.cols, numel);
  if ((w.kind == WeightSlot::MATRIX || w.kind == WeightSlot::MATRIX_T || w.kind == WeightSlot::ROWS_BF16) && ndim >= 2 &&
      shape[0] != w.rows)
    return fail(c, "ccb_load_weight(%s): expected leading dimension %lld, got %lld", name, w.rows, static_cast<long long>(shape[0]));
  int r = 0;
  switch (w.kind) {
    case WeightSlot::MATRIX:
    case WeightSlot::ROWS_BF16:
      r = convert_rows_bf16(dev_ptr, dtype, w.rows, static_cast<int>(w.cols), static_cast<bf16*>(w.dst), w.dst_ld, s);
      break;
    case WeightSlot::MATRIX_T:
      r = transpose_bf16(dev_ptr, dtype, static_cast<int>(w.rows), static_cast<int>(w.cols), static_cast<bf16*>(w.dst), w.dst_ld, s);
      break;
    case WeightSlot::VECTOR_F32:
      r = convert_f32(dev_ptr, dtype, w.rows * w.cols, static_cast<float*>(w.dst), s);
      break;
  }
  if (r != 0) return fail(c, "ccb_load_weight(%s): conversion kernel failed: %s", name, cudaGetErrorString(static_cast<cudaError_t>(r)));
  c->launches++;
  w.loaded = true;
  if (w.flag) *w.flag = true;
  return 0;
}

int ccb_weights_complete(ccb_ctx* c) {
  if (!c) return -1;
  DeviceGuard dev_guard(c->device);
  for (auto& kvp : c->slots)
    if (!kvp.second.loaded && !kvp.second.optional) return fail(c, "weight not loaded: %s", kvp.first.c_str());
  return 0;
}

int64_t ccb_preprocess_scratch_bytes(int H, int W, int new_h, int new_w, int n_px) {
  return static_cast<int64_t>(preprocess_scratch_bytes(H, W, new_h, new_w, n_px));
}

int ccb_preprocess_image(ccb_ctx* c, const uint8_t* rgb_hwc, int H, int W, int new_h, int new_w, int crop_top, int crop_left,
                         int n_px, const float* mean3, const float* std3, float* out_chw, void* scratch, int64_t scratch_bytes,
                         void* stream) {
  if (!c || !rgb_hwc || !mean3 || !std3 || !out_chw || !scratch) return fail(c, "ccb_preprocess_image: null argument");
  DeviceGuard dev_guard(c->device);
  const int r = preprocess_image(rgb_hwc, H, W, new_h, new_w, crop_top, crop_left, n_px, mean3, std3, out_chw, scratch,
                                 static_cast<size_t>(scratch_bytes), static_cast<cudaStream_t>(stream));
  if (r != 0) return fail(c, "ccb_preprocess_image: bad geometry / scratch too small / launch failed (%d)", r);
  c->launches += (new_h == H && new_w == W) ? 1 : 4;
  return 0;
}

int ccb_vit_encode(ccb_ctx* c, const void* images, int dtype, int B, float* feat_out, void* stream) {
  if (!c || !images || !feat_out) return fail(c, "ccb_vit_encode: null argument");
  DeviceGuard dev_guard(c->device);
  return vit_forward(c, images, dtype, B, feat_out, static_cast<cudaStream_t>(stream));
}

int ccb_vit_encode_tokens(ccb_ctx* c, const void* images, int dtype, int B, float* tokens_out, void* stream) {
  if (!c || !images || !tokens_out) return fail(c, "ccb_vit_encode_tokens: null argument");
  DeviceGuard dev_guard(c->device);
  return vit_forward(c, images, dtype, B, tokens_out, static_cast<cudaStream_t>(stream), true);
}

int ccb_clip_encode_text(ccb_ctx* c, const int32_t* tokens, int B, float* feat_out, void* stream) {
  if (!c || !tokens || !feat_out) return fail(c, "ccb_clip_encode_text: null argument");
  DeviceGuard dev_guard(c->device);
  return text_forward(c, tokens, B, feat_out, static_cast<cudaStream_t>(stream));
}

int ccb_map_prefix(ccb_ctx* c, const float* feat, int B, float* prefix_out, void* stream) {
  if (!c || !feat || !prefix_out) return fail(c, "ccb_map_prefix: null argument");
  DeviceGuard dev_guard(c->device);
  return map_forward(c, feat, B, prefix_out, c->desc.map_prefix_len, static_cast<cudaStream_t>(stream));
}

int ccb_embed_tokens(ccb_ctx* c, const int32_t* tokens, int n, float* out, void* stream) {
  if (!c || !tokens || !out) return fail(c, "ccb_embed_tokens: null argument");
  DeviceGuard dev_guard(c->device);
  if (n <= 0) return 0;
  RUN(embed_tokens(c->wte, nullptr, tokens, nullptr, out, n, c->desc.lm_d, c->desc.lm_vocab, 1, static_cast<cudaStream_t>(stream)));
  return 0;
}

int ccb_lm_forward(ccb_ctx* c, const float* embeds, int B, int S, const uint8_t* key_mask, float* logits_out,
                   int64_t ld_logits, int last_only, void* stream) {
  if (!c || !embeds || !logits_out) return fail(c, "ccb_lm_forward: null argument");
  DeviceGuard dev_guard(c->device);
  if (B <= 0 || S <= 0 || static_cast<long long>(B) * S > c->desc.max_lm_tokens)
    return fail(c, "ccb_lm_forward: B*S=%lld exceeds max_lm_tokens=%d", static_cast<long long>(B) * S, c->desc.max_lm_tokens);
  if (const char* why = attention_prefill_unsupported(S, c->desc.lm_d / c->desc.lm_heads, 1, false, c->desc.lm_rotary_dim, key_mask != nullptr))
    return fail(c, "ccb_lm_forward: S=%d with head_dim %d: %s", S, c->desc.lm_d / c->desc.lm_heads, why);
  if (c->desc.lm_arch == CCB_LM_GPT2 && S > c->desc.lm_n_pos)
    return fail(c, "ccb_lm_forward: S=%d exceeds the model's %d learned positions", S, c->desc.lm_n_pos);
  if (ld_logits < c->desc.lm_vocab) return fail(c, "ccb_lm_forward: ld_logits < vocab");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (lm_prefill_layers(c, embeds, B, S, key_mask, false, s)) return -1;
  return lm_logits(c, B, S, last_only, logits_out, ld_logits, s);
}

int ccb_generate(ccb_ctx* c, const ccb_gen_params* p, const float* embeds, int N, int S0, int32_t* tokens_out,
                 int32_t* lengths_out, float* scores_out, void* stream) {
  if (!c || !p || !embeds || !tokens_out) return fail(c, "ccb_generate: null argument");
  DeviceGuard dev_guard(c->device);
  cudaStream_t caller = static_cast<cudaStream_t>(stream);
  if (fence_in(c, caller)) return -1;
  const int r = generate_on_work_stream(c, p, embeds, N, S0, tokens_out, lengths_out, scores_out);
  if (fence_out(c, caller)) return -1;
  return r;
}

int ccb_caption_images(ccb_ctx* c, const ccb_gen_params* p, const void* images, int dtype, int N, int append_bos,
                       int32_t* tokens_out, int32_t* lengths_out, float* scores_out, void* stream) {
  if (!c || !p || !images || !tokens_out) return fail(c, "ccb_caption_images: null argument");
  DeviceGuard dev_guard(c->device);
  cudaStream_t caller = static_cast<cudaStream_t>(stream);
  if (fence_in(c, caller)) return -1;
  cudaStream_t s = c->work;
  const int P = c->desc.map_prefix_len, d = c->desc.lm_d;
  const int extra = append_bos >= 0 ? 1 : 0;
  const bool all_tokens = c->desc.map_kind == CCB_MAP_TRANSFORMER_ALL;
  if (all_tokens && c->desc.vit_present && c->desc.map_clip_len != (c->desc.vit_image / c->desc.vit_patch) * (c->desc.vit_image / c->desc.vit_patch) + 1)
    return fail(c, "ccb_caption_images: map_clip_len=%d does not match the ViT's token count", c->desc.map_clip_len);
  int r = vit_forward(c, images, dtype, N, c->feat, s, all_tokens);
  if (r == 0) r = map_forward(c, c->feat, N, c->prefix, P + extra, s);
  if (r == 0 && extra) {
    if (append_bos >= c->desc.lm_vocab) {
      r = fail(c, "ccb_caption_images: BOS id %d outside the vocabulary", append_bos);
    } else {
      token_rows_kernel<<<N, 256, 0, s>>>(c->wte, append_bos, c->prefix, static_cast<long long>(P + extra) * d, P, d);
      const int lc = launch_check();
      if (lc) r = fail(c, "token_rows_kernel: %s", cudaGetErrorString(static_cast<cudaError_t>(lc)));
      else c->launches++;
    }
  }
  if (r == 0) r = generate_on_work_stream(c, p, c->prefix, N, P + extra, tokens_out, lengths_out, scores_out);
  if (fence_out(c, caller)) return -1;
  return r;
}

int ccb_timing_sum(ccb_ctx* c, int n_calls, float* prefill_ms, float* decode_ms, int* decode_steps) {
  if (!c) return -1;
  DeviceGuard dev_guard(c->device);
  if (n_calls <= 0 || n_calls > ccb_ctx::kTimingSlots || n_calls > c->generate_calls)
    return fail(c, "ccb_timing_sum: n_calls=%d outside [1, min(%d, generate calls so far = %lld)]", n_calls,
                ccb_ctx::kTimingSlots, c->generate_calls);
  float a = 0.f, b = 0.f;
  int steps = 0;
  for (int i = 1; i <= n_calls; ++i) {
    const int slot = static_cast<int>((c->generate_calls - i) % ccb_ctx::kTimingSlots);
    float x = 0.f, y = 0.f;
    CUDA_OK(cudaEventElapsedTime(&x, c->ev_t0[slot], c->ev_t1[slot]));
    CUDA_OK(cudaEventElapsedTime(&y, c->ev_t1[slot], c->ev_t2[slot]));
    a += x;
    b += y;
    steps += c->timing_steps[slot];
  }
  if (prefill_ms) *prefill_ms = a;
  if (decode_ms) *decode_ms = b;
  if (decode_steps) *decode_steps = steps;
  return 0;
}

int ccb_last_timing(ccb_ctx* c, float* prefill_ms, float* decode_ms, int* decode_steps) {
  if (!c) return -1;
  DeviceGuard dev_guard(c->device);
  return ccb_timing_sum(c, 1, prefill_ms, decode_ms, decode_steps);
}

// ---------------------------------------------------------------------------------- samplers on caller tensors
int ccb_sample(ccb_ctx* c, const float* logits, int64_t ld, int B, int V, const ccb_gen_params* p,
               const int32_t* history, int64_t ld_hist, int hist_len, int step, float* filtered_out, int32_t* next_out,
               int32_t* alt_out, void* stream) {
  if (!c || !logits || !p || !next_out) return fail(c, "ccb_sample: null argument");
  DeviceGuard dev_guard(c->device);
  SampleParams sp = sample_params(c, p, B);
  sp.history = history;
  sp.ld_hist = ld_hist;
  sp.hist_len_scalar = hist_len;
  sp.step_scalar = step;
  sp.q_step_stride = 0;  // q_noise here is the [B, q_ld] draw of this one step
  sp.filtered_out = filtered_out;
  sp.alt_out = alt_out;
  RUN(sample_top_p(logits, ld, B, V, sp, next_out, static_cast<cudaStream_t>(stream)));
  return 0;
}

int ccb_argmax(ccb_ctx* c, const float* logits, int64_t ld, int B, int V, int32_t* next_out, void* stream) {
  if (!c || !logits || !next_out) return fail(c, "ccb_argmax: null argument");
  DeviceGuard dev_guard(c->device);
  RUN(sample_greedy(logits, ld, B, V, next_out, static_cast<cudaStream_t>(stream)));
  return 0;
}

int ccb_cross_entropy(ccb_ctx* c, const float* logits, int64_t ld, int rows, int V, const int32_t* targets,
                      const int32_t* row_map, int ignore_index, float* row_loss, float* loss_out, void* stream) {
  if (!c || !logits || !targets || !row_loss || !loss_out) return fail(c, "ccb_cross_entropy: null argument");
  DeviceGuard dev_guard(c->device);
  if (rows <= 0 || V <= 0 || ld < V) return fail(c, "ccb_cross_entropy: rows=%d V=%d ld=%lld", rows, V, static_cast<long long>(ld));
  RUN(cross_entropy(logits, ld, rows, V, targets, row_map, ignore_index, row_loss, loss_out, static_cast<cudaStream_t>(stream)));
  c->launches++;   // (two kernels)
  return 0;
}

int ccb_beam_step(ccb_ctx* c, const float* logits, int64_t ld, int N, int beam, int V, float temperature,
                  int stop_token, int step, float* scores, float* seq_lengths, uint8_t* has_stopped, int32_t* tokens,
                  int max_len, int32_t* next_tokens, int32_t* src_rows, void* stream) {
  if (!c || !logits || !scores || !seq_lengths || !has_stopped || !tokens || !next_tokens || !src_rows)
    return fail(c, "ccb_beam_step: null argument");
  DeviceGuard dev_guard(c->device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  // the step counter lives in device memory for the graph-replayed loop; stage the caller's value
  CUDA_OK(cudaMemcpyAsync(c->step, &step, sizeof(int), cudaMemcpyHostToDevice, s));
  CUDA_OK(cudaStreamSynchronize(s));  // `step` is a stack variable
  BeamState st;
  st.scores = scores;
  st.seq_lengths = seq_lengths;
  st.has_stopped = has_stopped;
  st.tokens = tokens;
  st.max_len = max_len;
  st.step = c->step;
  st.cand_scratch = c->beam_cand;
  st.cand_rows = c->max_rows;
  if (N * beam > c->max_rows) return fail(c, "ccb_beam_step: N * beam = %d exceeds the context's %d rows", N * beam, c->max_rows);
  c->launches++;   // (two kernels)
  RUN(beam_step(logits, ld, N, beam, V, temperature, stop_token, st, next_tokens, src_rows, nullptr, 0, nullptr, s));
  return 0;
}

// ---------------------------------------------------------------------------------- single operators
int ccb_op_linear(ccb_ctx* c, const void* x, int64_t lda, int tokens, const void* w, int features, int K,
                  const float* bias, int act, const float* residual, int64_t ldr, void* out, int64_t ldo, int out_bf16,
                  int orientation, int bn, int split_k, void* stream) {
  return ccb_op_linear_ex(c, x, lda, tokens, w, 0, features, K, bias, act, residual, ldr, out, ldo, out_bf16, 0, 0, 0,
                          orientation, bn, split_k, stream);
}

int ccb_op_linear_ex(ccb_ctx* c, const void* x, int64_t lda, int tokens, const void* w, int64_t ldw, int features, int K,
                     const float* bias, int act, const float* residual, int64_t ldr, void* out, int64_t ldo, int out_bf16,
                     int rg_in, int rg_out, int rg_off, int orientation, int bn, int split_k, void* stream) {
  if (!c || !x || !w || !out) return fail(c, "ccb_op_linear: null argument");
  DeviceGuard dev_guard(c->device);
  GemmArgs g;
  g.act = static_cast<const bf16*>(x);
  g.lda = lda;
  g.tokens = tokens;
  g.weight = static_cast<const bf16*>(w);
  g.ldw = ldw;
  g.rg_in = rg_in;
  g.rg_out = rg_out;
  g.rg_off = rg_off;
  g.features = features;
  g.K = K;
  g.bias = bias;
  g.act_fn = act;
  g.residual = residual;
  g.ldr = ldr;
  g.out = out;
  g.ldo = ldo;
  g.out_bf16 = out_bf16;
  g.force_orientation = orientation;
  g.force_bn = bn;
  g.force_split = split_k;
  static const bool op_pdl = [] {   // tuning (tools/bench_stream.py): chain back-to-back operator launches like the engine does
    const char* e = getenv("CCB_OP_PDL");
    return e && e[0] == '1';
  }();
  g.allow_pdl = op_pdl ? 1 : 0;
  RUN(gemm_launch(g, c->gemm_ws, static_cast<cudaStream_t>(stream)));
  return 0;
}

int ccb_debug_gemm_trace(ccb_ctx* c, void* trace_u64, int64_t stride_u64, int launches) {
  if (!c) return -1;
  c->gemm_ws.trace = static_cast<unsigned long long*>(trace_u64);
  c->gemm_ws.trace_stride = stride_u64;
  c->gemm_ws.trace_launches = launches > 0 ? launches : 1;
  c->gemm_ws.trace_count = 0;
  return 0;
}

int ccb_debug_set_mega(ccb_ctx* c, int enable) {
  if (!c) return -1;
  c->mega.enabled = enable != 0;   // 0: operator chain, otherwise the persistent kernel
  return c->mega.available ? 1 : 0;
}

int ccb_debug_copy_buffer(ccb_ctx* c, int which, void* dst, int64_t bytes, void* stream) {
  if (!c || !dst) return -1;
  DeviceGuard dev_guard(c->device);
  const void* src = nullptr;
  int64_t size = -1;   // known for the KV pool and the block table
  switch (which) {
    case 0: src = c->h; break;
    case 1: src = c->x; break;
    case 2: src = c->att; break;
    case 3: src = c->mlp; break;
    case 4: src = c->logits; break;
    case 5: src = c->qkv; break;
    case 6: src = c->kv.base; size = static_cast<int64_t>(2) * c->desc.lm_layers * c->kv_pool_tokens * c->desc.lm_d * sizeof(bf16); break;
    case 7: src = c->block_table; size = static_cast<int64_t>(c->max_rows) * c->max_pages_per_row * sizeof(int); break;
    default: return fail(c, "ccb_debug_copy_buffer: unknown buffer %d", which);
  }
  if (size >= 0 && (bytes < 0 || bytes > size))
    return fail(c, "ccb_debug_copy_buffer: %lld bytes requested from buffer %d of %lld bytes", static_cast<long long>(bytes), which,
                static_cast<long long>(size));
  CUDA_OK(cudaMemcpyAsync(dst, src, static_cast<size_t>(bytes), cudaMemcpyDeviceToDevice, static_cast<cudaStream_t>(stream)));
  return 0;
}

int ccb_debug_kv_layout(ccb_ctx* c, int64_t out[6]) {
  if (!c || !out) return fail(c, "ccb_debug_kv_layout: null argument");
  if (c->kv.page_tokens <= 0) return fail(c, "ccb_debug_kv_layout: no generate call yet");
  const KvCache& k = c->kv;
  const int64_t v[6] = {k.L, k.H, k.hd, k.page_tokens, k.num_pages, k.max_pages_per_row};
  for (int i = 0; i < 6; ++i) out[i] = v[i];
  return 0;
}

int ccb_debug_mega_trace(ccb_ctx* c, void* trace_u64) {
  if (!c) return -1;
  c->mega.trace = static_cast<unsigned long long*>(trace_u64);
  return c->mega.available ? c->mega.ncta : 0;
}

int ccb_op_layernorm(ccb_ctx* c, const float* x, const float* gamma, const float* beta, float eps, void* y_bf16,
                     int rows, int d, void* stream) {
  if (!c || !x || !gamma || !beta || !y_bf16) return fail(c, "ccb_op_layernorm: null argument");
  DeviceGuard dev_guard(c->device);
  RUN(layernorm_f32_bf16(x, d, gamma, beta, eps, static_cast<bf16*>(y_bf16), d, rows, d, static_cast<cudaStream_t>(stream)));
  return 0;
}

int ccb_op_attention(ccb_ctx* c, const void* qkv_bf16, void* out_bf16, int B, int S, int H, int hd, float scale,
                     int causal, int rotary_dim, void* stream) {
  if (!c || !qkv_bf16 || !out_bf16) return fail(c, "ccb_op_attention: null argument");
  DeviceGuard dev_guard(c->device);
  RUN(attention_prefill(static_cast<const bf16*>(qkv_bf16), static_cast<bf16*>(out_bf16), B, S, H, hd, scale, causal,
                        nullptr, 0, nullptr, 0, rotary_dim, nullptr, static_cast<cudaStream_t>(stream)));
  return 0;
}

int ccb_op_attention_decode(ccb_ctx* c, const void* qkv_bf16, void* out_bf16, int64_t ldo, int rows, int H, int hd, float scale,
                            void* kv_bf16, int layers, int layer, int num_pages, int page_tokens, int max_pages_per_row,
                            const int32_t* block_table, const int32_t* ctx_len, int rotary_dim, void* stream) {
  if (!c || !qkv_bf16 || !out_bf16 || !kv_bf16 || !block_table || !ctx_len)
    return fail(c, "ccb_op_attention_decode: null argument");
  if (layers <= 0 || layer < 0 || layer >= layers) return fail(c, "ccb_op_attention_decode: layer %d outside [0, %d)", layer, layers);
  if (page_tokens <= 0 || num_pages <= 0 || max_pages_per_row <= 0)
    return fail(c, "ccb_op_attention_decode: page_tokens=%d, num_pages=%d, max_pages_per_row=%d must be positive", page_tokens,
                num_pages, max_pages_per_row);
  if (hd != 64 && hd != 128 && hd != 256) return fail(c, "ccb_op_attention_decode: head_dim %d unsupported (64/128/256)", hd);
  if (rows < 0 || H <= 0) return fail(c, "ccb_op_attention_decode: rows=%d, H=%d", rows, H);
  DeviceGuard dev_guard(c->device);
  KvCache kv;
  kv.base = static_cast<bf16*>(kv_bf16);
  kv.L = layers;
  kv.H = H;
  kv.hd = hd;
  kv.page_tokens = page_tokens;
  kv.num_pages = num_pages;
  kv.max_pages_per_row = max_pages_per_row;
  RUN(attention_decode(static_cast<const bf16*>(qkv_bf16), static_cast<bf16*>(out_bf16), ldo, rows, H, hd, scale, &kv, layer,
                       block_table, ctx_len, rotary_dim, static_cast<cudaStream_t>(stream)));
  return 0;
}

}  // extern "C"
