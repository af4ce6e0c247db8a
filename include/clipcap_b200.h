/* libclipcap_b200 -- C ABI of the B200-native caption-generation hot path.
 *
 * The reference (andreaskoepf/CLIP-Image-Captioning) is pure Python and has no FFI: its boundary for this path
 * is the Python attribute surface listed in SURVEY.md section 8(b).  Each entry point below names the reference
 * call it replaces (file:line in the reference tree); the Python host code in clip-image-captioning_b200/
 * keeps the reference names/signatures and forwards to these functions through ctypes (see INTEGRATION.md).
 *
 * Conventions
 *   - return value 0 = OK, negative = error; ccb_last_error(ctx) (or ccb_last_error(NULL) for ccb_create
 *     failures) returns a human-readable message.  No C++ exception crosses the ABI.
 *   - every data pointer is a DEVICE pointer to a contiguous row-major tensor owned by the caller (PyTorch);
 *     the library never frees caller memory and allocates only inside ccb_create.
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*); no host synchronisation except
 *     where stated (ccb_caption_dataset, ccb_caption_dataset_beam, ccb_beam_step).  A ccb_ctx is bound to one device and is not thread-safe (one ctx per rank / GPU).
 *   - there is no CPU fallback: without an sm_100 device ccb_create fails.
 */
#ifndef CLIPCAP_B200_H_
#define CLIPCAP_B200_H_

#include <stdint.h>

#if defined(__GNUC__)
#define CCB_API __attribute__((visibility("default")))
#else
#define CCB_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ccb_ctx ccb_ctx;

enum { CCB_DTYPE_F32 = 0, CCB_DTYPE_F16 = 1, CCB_DTYPE_BF16 = 2 };
enum { CCB_LM_GPT2 = 0, CCB_LM_GPTJ = 1 };
/* TRANSFORMER_ALL: layers/Transformer.py:164-203 (TransformerMapperAllFeatures: one mapper token per ViT token, the
 * fork's default training configuration, train.py:73 use_all_vit_features=True) */
enum { CCB_MAP_NONE = 0, CCB_MAP_TRANSFORMER = 1, CCB_MAP_MLP = 2, CCB_MAP_TRANSFORMER_ALL = 3 };
/* activation codes (mapper act_fn_name, layers/Transformer.py:117-130; ViT QuickGELU; GPT gelu_new) */
enum {
  CCB_ACT_NONE = 0, CCB_ACT_RELU = 1, CCB_ACT_QUICKGELU = 2, CCB_ACT_GELU_NEW = 3, CCB_ACT_GELU = 4,
  CCB_ACT_ELU = 5, CCB_ACT_SELU = 6, CCB_ACT_TANH = 7,
  CCB_ACT_GEGLU = 8   /* mapper MLP only (layers/Transformer.py:74,112-114): fc1 is 2 x hidden wide, x * gelu(gate) */
};
enum { CCB_GEN_GREEDY = 0, CCB_GEN_SAMPLE = 1, CCB_GEN_BEAM = 2 };

typedef struct ccb_model_desc {
  /* language model: lms/GPT2.py:6-19 (HF GPT2LMHeadModel) or lms/GPTJ.py:5-18 (HF GPTJForCausalLM) */
  int32_t lm_arch, lm_d, lm_layers, lm_heads, lm_vocab, lm_n_pos, lm_rotary_dim;
  float lm_ln_eps;
  /* prefix mapper: layers/Transformer.py:133-161 (TransformerMapper); MLP = upstream ClipCap MLP mapper;
   * TRANSFORMER_ALL: map_clip_len = number of ViT tokens (50 for ViT-B/32 @ 224), optional pos_embeddings */
  int32_t map_kind, map_dim_clip, map_clip_len, map_prefix_len, map_heads, map_layers, map_hidden, map_act;
  /* image encoder: OpenAI CLIP VisionTransformer (call sites inference.py:311, evaluate_model.py:359) */
  int32_t vit_present, vit_image, vit_patch, vit_width, vit_layers, vit_heads, vit_out;
  /* capacity */
  int32_t max_images;      /* images (sequences before beam expansion) per call */
  int32_t max_beam;        /* >= 1 */
  int32_t max_ctx;         /* prefix + generated tokens per sequence */
  int32_t max_lm_tokens;   /* max B*S of one ccb_lm_forward call */
  int32_t page_tokens;     /* KV page size for greedy / sampling (beam search uses token-granular pages) */
  /* CLIP text tower for re-ranking (clip_model.encode_text: sampling.py:31, evaluate_model.py:182-352; OpenAI
   * clip/model.py CLIP.encode_text): vocab 49408, context 77, width 512, 12 layers, 8 heads, output 512 for ViT-B/32 */
  int32_t text_present, text_vocab, text_ctx, text_width, text_layers, text_heads, text_out;
  int32_t max_texts;       /* token sequences per ccb_clip_encode_text call */
} ccb_model_desc;

typedef struct ccb_gen_params {
  int32_t mode;              /* CCB_GEN_* */
  int32_t max_new_tokens;    /* entry_length (inference.py:77) / max_decode_length (evaluate_model.py:109) */
  int32_t stop_token;        /* tokenizer.encode('.')[0] = 13 for GPT-2; < 0 disables stopping */
  int32_t max_stops;         /* 1 = inference.py:284; 3 = evaluate_model.py:169-172 */
  int32_t eos_token;         /* special id that always terminates (evaluate_model.py:171); < 0 = none */
  float temperature;
  float top_p;               /* <= 0 disables */
  int32_t top_k;             /* <= 0 disables */
  float repetition_penalty;  /* 1.0 disables (inference.py:53-57) */
  int32_t beam_size;         /* inference.py:76 */
  uint64_t seed;             /* Philox seed when q_noise == NULL */
  const float* q_noise;      /* optional Exp(1) noise [max_new_tokens, N, q_ld] (torch.multinomial contract) */
  int64_t q_ld;
  const int64_t* row_ids;    /* optional global image ids [N] keying the Philox stream (multi-GPU invariance) */
  const float* top_p_rows;   /* optional per-row top_p [N] (sampling.py:146-148) */
  const int32_t* top_k_rows; /* optional per-row top_k [N] (sampling.py:135-145) */
  float typ_p;               /* typical decoding budget (sampling.py:72-102, applied after top-k / top-p as in
                                sampling.py:205-206); <= 0 disables */
  const float* typ_p_rows;   /* optional per-row budgets [N]: the filter then runs on every row, as the reference does
                                when any(typ_p > 0) */
} ccb_gen_params;

/* ---- lifetime ------------------------------------------------------------------------------------------ */
CCB_API int ccb_create(ccb_ctx** out, const ccb_model_desc* desc, int device);
CCB_API void ccb_destroy(ccb_ctx* ctx);
CCB_API const char* ccb_last_error(const ccb_ctx* ctx);
/* bytes of device memory held by the context (weights + KV pages + workspaces) */
CCB_API int64_t ccb_device_bytes(const ccb_ctx* ctx);

/* ---- weights ------------------------------------------------------------------------------------------- */
/* Ingest one state_dict tensor (names as in SURVEY.md appendix B.3 under "clip_project.", "language_model.",
 * "visual_encoder." / "visual."): copies + repacks to bf16 K-major (Conv1D [in,out] is transposed), LN / bias
 * to f32.  The caller keeps its tensor.  Returns 1 if the name is not used by this context (ignored). */
CCB_API int ccb_load_weight(ccb_ctx* ctx, const char* name, const void* dev_ptr, int dtype, const int64_t* shape, int ndim,
                    void* stream);
/* 0 when every weight the context needs has been loaded; otherwise -1 and ccb_last_error names one missing */
CCB_API int ccb_weights_complete(ccb_ctx* ctx);

/* ---- the step in front of the path: CLIP's image preprocessing ------------------------------------------ */
/* `clip_preprocess(image)` (clip.load(...)[1] = Compose([Resize(n_px, BICUBIC), CenterCrop(n_px), ToTensor, Normalize]);
 * applied at inference.py:310, evaluate_model.py:458-463; the same pipeline as blip_test.py:22-26) for ONE decoded RGB
 * image already on the device: rgb_hwc uint8 [H, W, 3] -> out_chw f32 [3, n_px, n_px].  PIL's antialiased bicubic resize
 * is reproduced exactly (Pillow Resample.c: double-precision coefficients rounded to 22-bit fixed point, uint8 between the
 * two passes).  The caller supplies the geometry exactly as torchvision computes it: the resized size (new_h, new_w) and
 * the crop origin.  mean3 / std3 are HOST pointers.  scratch: device memory of ccb_preprocess_scratch_bytes(...) bytes. */
CCB_API int64_t ccb_preprocess_scratch_bytes(int H, int W, int new_h, int new_w, int n_px);
CCB_API int ccb_preprocess_image(ccb_ctx* ctx, const uint8_t* rgb_hwc, int H, int W, int new_h, int new_w, int crop_top,
                                 int crop_left, int n_px, const float* mean3, const float* std3, float* out_chw, void* scratch,
                                 int64_t scratch_bytes, void* stream);

/* ---- the hot path, stage by stage ---------------------------------------------------------------------- */
/* clip_model.encode_image(image) (inference.py:311) / model.visual_encoder(image_tensor)
 * (evaluate_model.py:359): images [B,3,H,W] NCHW -> feat_out [B, vit_out] f32 */
CCB_API int ccb_vit_encode(ccb_ctx* ctx, const void* images, int dtype, int B, float* feat_out, void* stream);
/* the patched VisionTransformer.forward of the all-features path (inference.py:421-444, evaluate_model.py: same patch):
 * no ln_post / CLS extraction, every token projected: images [B,3,H,W] -> tokens_out [B, 1 + (H/patch)^2, vit_out] f32 */
CCB_API int ccb_vit_encode_tokens(ccb_ctx* ctx, const void* images, int dtype, int B, float* tokens_out, void* stream);
/* clip_model.encode_text(clip.tokenize(txt)) (sampling.py:30-31; OpenAI clip/model.py CLIP.encode_text): tokens [B, text_ctx]
 * int32 (the end-of-text token has the highest id, its position is where the features are read) -> feat_out [B, text_out]
 * f32, un-normalised like the reference (cos_sim, sampling.py:14-18, normalises). */
CCB_API int ccb_clip_encode_text(ccb_ctx* ctx, const int32_t* tokens, int B, float* feat_out, void* stream);
/* model.clip_project(prefix) (inference.py:312, model.py:137; layers/Transformer.py:153-161):
 * feat [B, map_dim_clip] f32 -> prefix_out [B, map_prefix_len, lm_d] f32.  With CCB_MAP_TRANSFORMER_ALL
 * (layers/Transformer.py:186-203) feat is [B, map_clip_len, map_dim_clip], the output of ccb_vit_encode_tokens. */
CCB_API int ccb_map_prefix(ccb_ctx* ctx, const float* feat, int B, float* prefix_out, void* stream);
/* language_model.get_embedding_text(tokens) (lms/GPT2.py:14-15): out [n, lm_d] f32 */
CCB_API int ccb_embed_tokens(ccb_ctx* ctx, const int32_t* tokens, int n, float* out, void* stream);
/* language_model.call(inputs_embeds=E[, attention_mask]) (lms/GPT2.py:17-19 -> HF forward):
 * embeds [B,S,lm_d] f32 -> logits [B,S,ld_logits] (last_only = 0) or [B,ld_logits] for the last position.
 * key_mask: optional [B,S] uint8 (1 = attend), the HF attention_mask on keys; NULL = no mask.
 * S is at most 256, and at most what the attention kernels hold at the LM's head_dim: 256 for head_dim 64 / 128
 * (GPT-2 family), 185 for head_dim 256 (GPT-J).  A longer S fails with a message naming S and head_dim before anything
 * is launched; the same limit applies to the prefix length S0 of ccb_generate / ccb_caption_images. */
CCB_API int ccb_lm_forward(ccb_ctx* ctx, const float* embeds, int B, int S, const uint8_t* key_mask, float* logits_out,
                   int64_t ld_logits, int last_only, void* stream);
/* generate_beam / generate_no_beam loops (inference.py:70-148, 219-292; evaluate_model.py:104-179), batched
 * per row, the whole loop on the device: embeds [N,S0,lm_d] f32 prefix embeddings (what the reference loops
 * receive as `embeds`, already including any text-prefix / BOS embedding).
 *   greedy / sample: tokens_out [N, max_new_tokens] int32, lengths_out [N], scores_out ignored (may be NULL)
 *   beam: tokens_out [N, beam, max_new_tokens], lengths_out [N, beam] (seq_lengths), scores_out [N, beam]
 *         (scores / seq_lengths, inference.py:138); the caller picks argmax like inference.py:143-144. */
CCB_API int ccb_generate(ccb_ctx* ctx, const ccb_gen_params* params, const float* embeds, int N, int S0, int32_t* tokens_out,
                 int32_t* lengths_out, float* scores_out, void* stream);
/* images -> captions in one call: ccb_vit_encode + ccb_map_prefix (+ BOS embedding appended when
 * append_bos >= 0, evaluate_model.py:124-133) + ccb_generate.  Same outputs as ccb_generate. */
CCB_API int ccb_caption_images(ccb_ctx* ctx, const ccb_gen_params* params, const void* images, int dtype, int N,
                       int append_bos, int32_t* tokens_out, int32_t* lengths_out, float* scores_out, void* stream);
/* A whole shard of images -> captions with continuous batching, greedy or sampling: `rows` decode slots stay busy, and a
 * slot whose caption has finished takes the next image.  images [n_images, 3, H, W] (device); tokens_out
 * [n_images, max_new_tokens] and lengths_out [n_images] in image order (device); *decode_steps_out (HOST) = decode steps run.
 * Per image, (tokens[:len], len) is what ccb_caption_images gives; unlike there, positions at or past a caption's length
 * are 0.  Sampling keys each image's Philox stream by (seed, first_row_id + image index, step), so the result depends
 * neither on `rows` nor on the order in which images are taken.
 * The call synchronises the host once per round of a few decode steps, to learn which slots have finished; it returns
 * once the last round has completed.  ccb_last_timing / ccb_timing_sum do not count it.
 * Rejected with a message, nothing launched: beam mode, q_noise, the per-row arrays (row_ids, top_p_rows, top_k_rows,
 * typ_p_rows), rows outside [1, max_images * max_beam], map_prefix_len (+ 1 with append_bos >= 0) + max_new_tokens above
 * max_ctx, and the prefix shapes ccb_caption_images rejects. */
CCB_API int ccb_caption_dataset(ccb_ctx* ctx, const ccb_gen_params* params, const void* images, int dtype, int n_images,
                                int rows, int append_bos, int64_t first_row_id, int32_t* tokens_out, int32_t* lengths_out,
                                int64_t* decode_steps_out, void* stream);
/* A whole shard of images -> beam-search captions with continuous batching (generate_beam, inference.py:70-148, per
 * image): `groups` images are in flight, each holding beam_size decode rows, and an image's group takes the next image
 * once all of its beams have stopped (the reference's `if has_stopped.all(): break`) or it has produced max_new_tokens
 * tokens.  images [n_images, 3, H, W] (device); in image order (device): tokens_out [n_images, beam, max_new_tokens] int32,
 * lengths_out [n_images, beam] (seq_lengths), scores_out [n_images, beam] (scores / seq_lengths, inference.py:138), the
 * layout of ccb_caption_images in beam mode: the caller picks argmax like inference.py:143-144.  Positions past a beam's
 * length are 0.  *decode_steps_out (HOST) = decode steps run.
 * The call synchronises the host once per round of a few decode steps, to learn which groups have finished; it returns
 * once the last round has completed.  ccb_last_timing / ccb_timing_sum do not count it.  max_stops, eos_token, seed
 * and the sampling fields are ignored, as ccb_generate ignores them in beam mode.
 * Rejected with a message, nothing launched: a mode other than beam, beam_size outside [1, min(max_beam, 8)], groups
 * outside [1, max_images], map_prefix_len (+ 1 with append_bos >= 0) + max_new_tokens above max_ctx, the prefix shapes
 * ccb_caption_images rejects, and beam_size * max(max_new_tokens, max_ctx) * 4 bytes above the 64 KB of shared memory
 * of the beam merge. */
CCB_API int ccb_caption_dataset_beam(ccb_ctx* ctx, const ccb_gen_params* params, const void* images, int dtype,
                                     int n_images, int groups, int append_bos, int32_t* tokens_out, int32_t* lengths_out,
                                     float* scores_out, int64_t* decode_steps_out, void* stream);
/* number of kernels launched by the library on this context since creation (CUDA-graph replays count the
 * kernels inside the graph) */
CCB_API int64_t ccb_launch_count(const ccb_ctx* ctx);
/* last generate call: device time (ms) of prefill and of the decode loop measured with events on `stream`;
 * valid after the stream has been synchronised. Returns 0 on success. */
CCB_API int ccb_last_timing(ccb_ctx* ctx, float* prefill_ms, float* decode_ms, int* decode_steps);
/* same, summed over the last n_calls generate calls (n_calls <= 64): total prefill ms, decode ms, decode steps */
CCB_API int ccb_timing_sum(ccb_ctx* ctx, int n_calls, float* prefill_ms, float* decode_ms, int* decode_steps);

/* ---- logit processors and samplers on caller tensors ---------------------------------------------------- */
/* sampling.py:114-162 top_k_top_p_filtering_batch (+ :65-69 repetition_penalty_apply, temperature) followed by
 * softmax + torch.multinomial(p, 1|2) == argmax(p / q).  logits [B, ld] f32 (not modified).
 * history [B, ld_hist] int32 with hist_len tokens per row (NULL = none).  q_noise [B, q_ld] or NULL (Philox).
 * filtered_out: optional [B, ld] f32 receiving the masked logits (-inf = removed).  next_out [B] int32;
 * alt_out optional [B] int32 = second draw without replacement (sampling.py:223). */
CCB_API int ccb_sample(ccb_ctx* ctx, const float* logits, int64_t ld, int B, int V, const ccb_gen_params* params,
               const int32_t* history, int64_t ld_hist, int hist_len, int step, float* filtered_out,
               int32_t* next_out, int32_t* alt_out, void* stream);
/* argmax with lowest-index tie rule (generate_beam with beam_size=1) */
CCB_API int ccb_argmax(ccb_ctx* ctx, const float* logits, int64_t ld, int B, int V, int32_t* next_out, void* stream);
/* teacher-forced loss: F.cross_entropy(logits.reshape(-1, V), tokens.flatten(), ignore_index=0) of
 * evaluate_model.py:511-514 (validation) and model.py:210-211 (training_step), forward only.  logits [*, ld] f32;
 * targets [rows] int32; row_map optional [rows] int32 = logits row of each target (the reference's
 * `logits[:, prefix_length-1:-1]` slice without a copy; NULL = row r); row_loss [rows] f32 out (0 for ignored rows);
 * loss_out [2] f32 = {mean over the rows with target != ignore_index (NaN if none), number of such rows}. */
CCB_API int ccb_cross_entropy(ccb_ctx* ctx, const float* logits, int64_t ld, int rows, int V, const int32_t* targets,
               const int32_t* row_map, int ignore_index, float* row_loss, float* loss_out, void* stream);
/* one beam-search step on caller state (inference.py:98-131): logits [N*beam, ld] (step 0: [N, ld]);
 * scores/seq_lengths [N,beam] f32, has_stopped [N,beam] uint8, tokens [N,beam,max_len] int32 updated in place;
 * next_tokens / src_rows [N*beam] int32 out.  N * beam must not exceed the context's rows (max_images * max_beam): the
 * rows' candidate lists are staged in a buffer of the context (two launches: rows, then the per-image merge). */
CCB_API int ccb_beam_step(ccb_ctx* ctx, const float* logits, int64_t ld, int N, int beam, int V, float temperature,
                  int stop_token, int step, float* scores, float* seq_lengths, uint8_t* has_stopped,
                  int32_t* tokens, int max_len, int32_t* next_tokens, int32_t* src_rows, void* stream);

/* ---- single operators on caller tensors (used by the parity tests and micro-benchmarks) ------------------ */
/* out[t, f] = act(sum_k x[t,k] * w[f,k] + bias[f]) + residual[t, f]; x [tokens, K] bf16 (ld lda), w [features, K]
 * bf16, bias f32 or NULL, residual f32 [tokens, ldr] or NULL, out f32 or bf16 [tokens, ldo].
 * orientation: 0 auto (swapped when tokens <= 256), 1 normal (tokens on the 128-row MMA side), 2 swapped (weights on the
 * 128-row side, tokens <= 256), 3 normal on the CTA-pair persistent kernel, 4 normal on the single-CTA persistent kernel.
 * bn: 0 auto, else the tile width in tokens (swapped) or features (normal).  split_k: 0 auto, else the number of K splits;
 * the swapped orientation only: with the normal orientation a non-zero split_k is an error. */
CCB_API int ccb_op_linear(ccb_ctx* ctx, const void* x, int64_t lda, int tokens, const void* w, int features, int K,
                  const float* bias, int act, const float* residual, int64_t ldr, void* out, int64_t ldo,
                  int out_bf16, int orientation, int bn, int split_k, void* stream);
/* ccb_op_linear with the addressing the engine's own GEMMs use (ccb_op_linear is this call with ldw = 0 and no remap):
 *   out[r(t), f] = act(sum_k x[t * lda + k] * w[f * ldw + k] + bias[f]) + residual[r(t) * ldr + f]
 *   r(t) = (t / rg_in) * rg_out + rg_off + t % rg_in   (identity when rg_in = rg_out = rg_off = 0)
 * out element (row r, column f) is at out + r * ldo + f.  ldw is the weight row pitch in elements (0: K), so w may be a
 * column range of a wider matrix.  residual may equal out (read before the element is written: an in-place residual
 * stream); no other overlap of out with x, w, bias or residual is allowed.  The row remap lays groups of rg_in token
 * rows into groups of rg_out output rows at offset rg_off (the all-features mapper's visual tokens inside each
 * sequence); it exists only in the normal orientation (orientation 1, 3 or 4, or 0 with tokens > 256).
 * Rejected with a message, nothing launched: act outside 0..7 (CCB_ACT_GEGLU is not an epilogue), K not a positive
 * multiple of 64, lda < K, ldw != 0 and ldw < K, ldo < features, a residual with ldr < features, a remap with
 * rg_in <= 0, rg_off < 0 or rg_off + rg_in > rg_out, x / w not 16-byte aligned or their row pitches not multiples of
 * 8 elements, and in the normal orientation out / residual / bias not 16-byte aligned.  The caller owns the extents:
 * x holds `tokens` rows, w `features` rows, out and residual every row r(t) for t < tokens. */
CCB_API int ccb_op_linear_ex(ccb_ctx* ctx, const void* x, int64_t lda, int tokens, const void* w, int64_t ldw, int features,
                  int K, const float* bias, int act, const float* residual, int64_t ldr, void* out, int64_t ldo,
                  int out_bf16, int rg_in, int rg_out, int rg_off, int orientation, int bn, int split_k, void* stream);
/* tuning aid, inert unless the library was built with -DCCB_TUNING (`python tools/build.py --tuning`): when non-NULL,
 * one-tile GEMM launch n of this context writes 8 globaltimer stamps per CTA to
 * trace[(n % launches) * stride_u64 + cta * 8 + k] (entry, setup, first tile landed, MMAs issued, accumulator ready,
 * cluster reduction reached, epilogue done, exit).  NULL (the default) disables it. */
CCB_API int ccb_debug_gemm_trace(ccb_ctx* ctx, void* trace_u64, int64_t stride_u64, int launches);
/* tuning aid for the persistent decode-step kernel (inert unless the library was built with -DCCB_TUNING,
 * `python tools/build.py --tuning`): when non-NULL every CTA writes globaltimer stamps of its phase
 * boundaries (grid-barrier waits / arrivals, in program order) to trace[cta * 2 * (8 * lm_layers + 2) + k].
 * Returns the number of CTAs of that kernel (0 when the model shape is not covered by it). */
CCB_API int ccb_debug_mega_trace(ccb_ctx* ctx, void* trace_u64);
/* A/B aid: 0 routes decode steps through the operator-per-kernel chain instead of the persistent kernel (CCB_MEGA=0 in
 * the environment); any other value (default) uses the persistent kernel.  Returns 1 when the persistent kernel covers
 * this model shape, else 0. */
CCB_API int ccb_debug_set_mega(ccb_ctx* ctx, int enable);
/* test aid: copies the first `bytes` of an internal buffer to `dst` (device memory) on `stream`:
 * 0 residual stream h (f32), 1 LayerNorm output x (bf16), 2 attention output (bf16), 3 MLP hidden (bf16),
 * 4 logits (f32, row pitch = vocab rounded up to 64), 5 fused qkv (bf16; operator-per-kernel decode only),
 * 6 KV pool (bf16 [layers][2][num_pages][heads][page_tokens][head_dim], geometry of ccb_debug_kv_layout),
 * 7 block table (int32 [max_images * max_beam][max_pages_per_row]).  For 6 and 7 more bytes than the buffer holds is an
 * error. */
CCB_API int ccb_debug_copy_buffer(ccb_ctx* ctx, int which, void* dst, int64_t bytes, void* stream);
/* test aid: the KV pool geometry of the last ccb_generate / ccb_caption_images call: out = {layers, heads, head_dim,
 * page_tokens, num_pages, max_pages_per_row}.  An error before the first such call. */
CCB_API int ccb_debug_kv_layout(ccb_ctx* ctx, int64_t out[6]);
/* y = LayerNorm(x) over the last dim: x f32 [rows, d] -> y bf16 [rows, d] */
CCB_API int ccb_op_layernorm(ccb_ctx* ctx, const float* x, const float* gamma, const float* beta, float eps, void* y_bf16,
                     int rows, int d, void* stream);
/* softmax(q k^T * scale [causal]) v for a fused qkv buffer [B*S, 3*H*hd] bf16 -> out [B*S, H*hd] bf16 */
CCB_API int ccb_op_attention(ccb_ctx* ctx, const void* qkv_bf16, void* out_bf16, int B, int S, int H, int hd, float scale,
                     int causal, int rotary_dim, void* stream);
/* One decode step of attention over a paged KV cache in caller memory, on the kernels the operator-per-kernel decode
 * chain runs (head_dim 64 / 128: one warp per (row, head); 256: one CTA per (row, head)).  qkv [rows, 3*H*hd] holds each
 * row's new token; row r attends over positions [0, ctx_len[r]] with the token at ctx_len[r] being the new one: its k
 * (GPT-J rotary at position ctx_len[r] on the first rotary_dim dims, as on q; 0 = none) and v are first stored into the
 * cache.  out row r starts at r * ldo (ldo >= H*hd, even).
 * kv [layers][2][num_pages][H][page_tokens][hd] (k then v); block_table [rows, max_pages_per_row]: position t of row r is
 * slot t % page_tokens of page block_table[r][t / page_tokens].  The caller keeps the contract the engine keeps:
 *   - every ctx_len[r] < max_pages_per_row (the engine's block table is sized for token-granular pages, and the kernels
 *     size their per-row score buffer and K/V tile from max_pages_per_row);
 *   - every page id that positions [0, ctx_len[r]] of row r use lies in [0, num_pages).
 * Null pointers, `layer` outside [0, layers), non-positive page geometry and an unsupported head_dim are rejected. */
CCB_API int ccb_op_attention_decode(ccb_ctx* ctx, const void* qkv_bf16, void* out_bf16, int64_t ldo, int rows, int H, int hd,
                                    float scale, void* kv_bf16, int layers, int layer, int num_pages, int page_tokens,
                                    int max_pages_per_row, const int32_t* block_table, const int32_t* ctx_len, int rotary_dim,
                                    void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CLIPCAP_B200_H_ */
