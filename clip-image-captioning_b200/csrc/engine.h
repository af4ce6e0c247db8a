// The context behind the C ABI: model description, packed weights, workspaces, the paged KV pool and the
// device-side generation state.  One ccb_ctx per GPU / rank; not thread-safe.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/clipcap_b200.h"
#include "internal.h"
#include "mega.h"

namespace ccb {

struct Linear {
  bf16* w = nullptr;      // [features, K] K-major
  float* bias = nullptr;  // [features] or null
  int features = 0, K = 0;
  bool has_bias = false;
  long long ldw = 0;      // row pitch in elements (0: K); wider for a view of a K-concatenated matrix
};
struct LayerNormW {
  float* g = nullptr;
  float* b = nullptr;
};
struct Block {            // one pre-LN transformer block (ViT / mapper / GPT-2 / GPT-J)
  LayerNormW ln1, ln2;
  Linear qkv, proj, fc, fc2;
  // GPT-J (parallel block): out_proj and fc_out are the column ranges [0, d) and [d, 5d) of ONE [d, 5d] matrix, so that the
  // decode step runs h += [att | gelu(fc_in)] . [W_out | W_fc_out]^T + b_fc_out as one weight-streaming GEMM (w == nullptr elsewhere)
  Linear projfc2;
};

// a weight the loader expects: where it goes and how the caller tensor is repacked
struct WeightSlot {
  enum Kind { MATRIX, MATRIX_T, VECTOR_F32, ROWS_BF16 } kind = MATRIX;
  void* dst = nullptr;     // bf16* (matrices) or float* (vectors)
  long long rows = 0;      // caller tensor logical [rows, cols] (after flattening trailing dims)
  long long cols = 0;
  long long dst_ld = 0;    // elements
  bool* flag = nullptr;    // set when loaded (optional biases)
  bool loaded = false;
  bool optional = false;
};

struct GraphEntry {
  cudaGraphExec_t exec = nullptr;
  int nodes = 0;
};

}  // namespace ccb

struct ccb_ctx {
  ccb_model_desc desc;
  int device = 0;
  int num_sms = 148;
  std::string err;

  // ---- device memory (everything is carved from a few cudaMalloc'd arenas in ccb_create)
  std::vector<void*> allocs;
  void* host_pinned = nullptr;    // cudaMallocHost'd: the continuous-batching ring below
  std::vector<size_t> alloc_sizes;
  int64_t device_bytes = 0;

  // ---- weights
  std::unordered_map<std::string, ccb::WeightSlot> slots;
  // language model
  ccb::bf16* wte = nullptr;       // [V, d]
  ccb::bf16* wpe = nullptr;       // [n_pos, d] (GPT-2)
  std::vector<ccb::Block> lm;
  ccb::LayerNormW lm_lnf;
  ccb::Linear lm_head;            // GPT-2: alias of wte (no bias); GPT-J: own weight + bias
  // mapper
  ccb::Linear map_linear;         // transformer mapper: [clip_len*d, dim_clip]; MLP mapper: first layer
  ccb::Linear map_mlp2;           // MLP mapper second layer
  float* map_pos = nullptr;          // TransformerMapperAllFeatures.pos_embeddings [clip_len, d] (optional)
  bool map_pos_present = false;
  float* map_prefix_const = nullptr;  // [P, d]
  std::vector<ccb::Block> mapper;
  // ViT
  ccb::Linear vit_conv;           // [width, 3*ps*ps]
  float* vit_cls = nullptr;
  float* vit_pos = nullptr;
  ccb::LayerNormW vit_ln_pre, vit_ln_post;
  std::vector<ccb::Block> vit;
  ccb::Linear vit_proj;           // [out, width]
  // CLIP text tower (re-ranking)
  ccb::bf16* txt_wte = nullptr;   // token_embedding [vocab, width]
  ccb::bf16* txt_wpe = nullptr;   // positional_embedding [ctx, width]
  std::vector<ccb::Block> txt;
  ccb::LayerNormW txt_ln_final;
  ccb::Linear txt_proj;           // text_projection [out, width]
  int* txt_positions = nullptr;   // [max_texts * ctx]: r % ctx
  int* txt_eot = nullptr;         // [max_texts]: argmax of the token ids of each sequence

  // ---- workspaces
  int max_rows_tokens = 0;        // rows of the activation workspaces
  int dmax = 0, hidden_max = 0;
  float* h = nullptr;             // residual stream f32 [M, dmax]
  ccb::bf16* x = nullptr;         // LN output / GEMM input bf16 [M, dmax]
  ccb::bf16* qkv = nullptr;       // [M, 3*dmax]
  ccb::bf16* att = nullptr;       // [M, dmax]
  ccb::bf16* mlp = nullptr;       // [M, hidden_max]
  ccb::bf16* attmlp = nullptr;    // GPT-J decode: [max_rows, 5 d] = [att | gelu(fc_in)], the fused GEMM's operand
  ccb::bf16* patches = nullptr;   // [B*np, 3*ps*ps]
  float* patch_emb = nullptr;     // [B*np, width]
  float* feat = nullptr;          // [B, vit_out] f32
  ccb::bf16* feat_bf16 = nullptr; // [B, dim_clip]
  float* prefix = nullptr;        // [B, P+1, d] f32 (mapper output + optional BOS embedding)
  float* logits = nullptr;        // [max_rows, ldv] f32
  int64_t ldv = 0;                // padded vocab row pitch
  ccb::GemmWorkspace gemm_ws;

  // ---- KV pool + generation state
  ccb::KvCache kv;                // page_tokens / num_pages are set per generate call
  long long kv_pool_tokens = 0;
  int max_rows = 0;               // max_images * max_beam
  int max_pages_per_row = 0;      // = max_ctx (token-granular worst case)
  int* block_table = nullptr;     // [max_rows, max_pages_per_row]
  int* block_table_prefill = nullptr;  // [max_images, max_pages_per_row]
  int* ctx_len = nullptr;         // [max_rows]
  int* step = nullptr;            // [1]
  int* next_tokens = nullptr;     // [max_rows]
  int* src_rows = nullptr;        // [max_rows]
  void* beam_cand = nullptr;      // [max_rows, kBeamCandPerRow] (value, flat index): beam_rows_kernel -> beam_merge_kernel
  int* gen_tokens = nullptr;      // [max_rows, max_ctx]
  int* lengths = nullptr;         // [max_rows]
  int* stops = nullptr;           // [max_rows]
  uint8_t* finished = nullptr;    // [max_rows]
  float* scores = nullptr;        // [max_rows]
  float* seq_lengths = nullptr;   // [max_rows]
  uint8_t* has_stopped = nullptr; // [max_rows]
  int* bos_token = nullptr;       // [max_images] scratch for the BOS embedding gather
  // continuous batching (ccb_caption_dataset): a slot (decode row) holds one image at a time; ccb_caption_dataset_beam
  // keeps the same per-unit state for its groups of beam rows (row_step = the group's beam steps)
  int* row_step = nullptr;        // [max_rows] tokens generated so far by the slot's image
  int* slot_image = nullptr;      // [max_rows] image index of the slot, -1 = none
  long long* slot_ids = nullptr;  // [max_rows] first_row_id + image index: the slot's Philox key
  int* refill_slots = nullptr;    // [max_rows] slots refilled at one round boundary, in refill order
  long long* refill_ids = nullptr;  // [max_images] Philox keys of one refill chunk's prefill rows
  int* refill_next = nullptr;     // [max_images] first tokens of one refill chunk
  void** cont_out = nullptr;      // [3] the caller's tokens / lengths (/ scores) outputs, read by the captured rounds
  // pinned host ring (two halves): per round the finished flags and images of the slots, per boundary the refill list
  uint8_t* h_finished = nullptr;  // [2, max_rows]
  int* h_slot_image = nullptr;    // [2, max_rows]
  int* h_refill = nullptr;        // [2, max_rows]
  cudaEvent_t ev_round[2] = {};

  // ---- persistent decode-step kernel (decode_mega.cu); unavailable -> operator-per-kernel decode step
  ccb::MegaState mega;

  // ---- streams / graphs / accounting
  cudaStream_t work = nullptr;
  cudaEvent_t ev_in = nullptr, ev_out = nullptr;
  // ring of (start, prefill done, decode done) events, one slot per generate call
  static constexpr int kTimingSlots = 64;
  cudaEvent_t ev_t0[kTimingSlots] = {}, ev_t1[kTimingSlots] = {}, ev_t2[kTimingSlots] = {};
  int timing_steps[kTimingSlots] = {};
  long long generate_calls = 0;
  std::unordered_map<std::string, ccb::GraphEntry> graphs;
  int64_t launches = 0;
  bool capturing = false;
  int capture_launches = 0;
};
