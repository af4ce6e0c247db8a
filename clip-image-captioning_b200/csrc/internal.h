// Internal (non-ABI) launch interface shared by the translation units of libclipcap_b200.so.
// Every launcher is asynchronous on `stream`, allocates nothing and returns a cudaError_t-compatible int
// (0 = ok).  Device pointers only.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace ccb {

typedef __nv_bfloat16 bf16;

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) is per DEVICE: "already configured" state is kept per device so that a
// second context on another GPU of the same process configures its kernels too.
constexpr int kMaxDevices = 64;
inline int current_device_slot() {
  int d = 0;
  cudaGetDevice(&d);
  return d >= 0 && d < kMaxDevices ? d : 0;
}

// Programmatic dependent launch for the kernels of the decode chain (they all call ptx::grid_dep_wait() before
// touching activations): CCB_PDL=0 in the environment switches it off.
bool pdl_enabled();

// <<<>>> with optional launch attributes (PDL).  Returns the launch status.
template <typename... KArgs, typename... Args>
inline cudaError_t launch_kernel(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, bool pdl,
                                 Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  if (pdl && pdl_enabled()) {
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
  }
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// ------------------------------------------------------------------ GEMM (gemm.cu)
struct GemmWorkspace {
  float* ws = nullptr;      // split-K partial tiles
  size_t ws_bytes = 0;
  int* sem = nullptr;       // per-tile semaphores (zero-initialised, self-resetting)
  int sem_count = 0;
  int num_sms = 148;
  // tuning only: per-CTA timelines; launch n writes to trace + (n % trace_launches) * trace_stride
  unsigned long long* trace = nullptr;
  long long trace_stride = 0;
  int trace_launches = 1;
  mutable long long trace_count = 0;
};

struct GemmArgs {
  const bf16* act = nullptr;   // [tokens, K] row-major, leading dim lda (elements)
  long long lda = 0;
  int tokens = 0;
  const bf16* weight = nullptr;  // [features, K] row-major (K-major), leading dim ldw (0: K)
  long long ldw = 0;
  int features = 0;
  int K = 0;                     // multiple of 64
  const float* bias = nullptr;   // [features] or null
  int act_fn = 0;                // ccb::Act
  const float* residual = nullptr;  // f32 [tokens(out rows), ldr] or null; may alias out
  long long ldr = 0;
  void* out = nullptr;           // [tokens(out rows), ldo]
  long long ldo = 0;
  int out_bf16 = 0;
  int rg_in = 0, rg_out = 0, rg_off = 0;  // out_row = (t / rg_in) * rg_out + rg_off + t % rg_in (0 = identity)
  // 0 auto (swapped when tokens <= 256), 1 normal (tokens on the 128-row MMA side: the persistent kernels, single-CTA or
  // CTA pair picked from the shape), 2 swapped (weights on the 128-row side: the one-tile-per-CTA kernel),
  // 3 normal on the CTA-pair persistent kernel, 4 normal on the single-CTA persistent kernel
  int force_orientation = 0;
  int force_bn = 0;              // 0 auto
  int force_split = 0;           // 0 auto; split-K exists in the swapped orientation only (an error otherwise)
  int allow_pdl = 0;             // 1: launched inside the engine's own chain (weights are never produced by the
                                 // preceding kernel, so their loads may start before the dependency wait)
};

int gemm_init(int device);  // resolves cuTensorMapEncodeTiled, sets smem attributes
int gemm_launch(const GemmArgs& a, const GemmWorkspace& w, cudaStream_t stream);
const char* gemm_last_error();

// ------------------------------------------------------------------ row-wise / glue kernels (rowwise.cu)
// y = LayerNorm(x) * gamma + beta, x f32 [rows, d] (leading dim ldx) -> y bf16 [rows, d] (leading dim ldy)
int layernorm_f32_bf16(const float* x, long long ldx, const float* gamma, const float* beta, float eps, bf16* y,
                       long long ldy, int rows, int d, cudaStream_t s);
// same but also writes the normalised row as f32 (final ViT ln_post -> proj input kept bf16; f32 copy for debug)
int layernorm_f32_f32(const float* x, long long ldx, const float* gamma, const float* beta, float eps, float* y,
                      long long ldy, int rows, int d, cudaStream_t s);
// ViT: NCHW image (f32 or f16 or bf16) -> im2col patches bf16 [B*gh*gw, 3*ps*ps] in conv-weight order (c, ky, kx), rows at
// pitch ldp >= 3*ps*ps (columns past 3*ps*ps are written as zeros)
int vit_patchify(const void* images, int img_dtype /*0 f32, 1 f16, 2 bf16*/, int B, int C, int H, int W, int ps,
                 bf16* patches, int ldp, cudaStream_t s);
// ViT: x[b,0,:] = cls + pos[0]; x[b,1+p,:] = patch_emb[b*np+p,:] + pos[1+p]; then ln_pre in place -> f32 stream
int vit_assemble_lnpre(const float* patch_emb, const float* cls, const float* pos, const float* g, const float* b,
                       float eps, float* x, int B, int np, int d, cudaStream_t s);
// mapper: seq[b, clip_len + p, :] = prefix_const[p, :]  (f32 stream [B, S, d]); rows [0, clip_len) are written
// by the `linear` GEMM epilogue.
int mapper_fill_const(const float* prefix_const, float* seq, int B, int clip_len, int P, int d, cudaStream_t s);
// all-features mapper: seq[b, t, :] = pos[t, :] (zeros when pos == null) for t < clip_len
int mapper_fill_pos(const float* pos, float* seq, int B, int clip_len, int P, int d, cudaStream_t s);
// f32 -> bf16 cast of a [rows, d] block (leading dims in elements)
int cast_f32_bf16(const float* x, long long ldx, bf16* y, long long ldy, int rows, int d, cudaStream_t s);
// geglu (layers/Transformer.py:112-114) in place: x[r, j] = x[r, j] * gelu(x[r, h + j]) for j < h, rows of pitch ldx >= 2h
int geglu_inplace(bf16* x, long long ldx, int rows, int h, cudaStream_t s);
// bf16/f32 embedding gather: h[r, :] = table[tok[r], :] (+ wpe[pos[r], :] if wpe) -> f32 [rows, d]
int embed_tokens(const bf16* wte, const bf16* wpe, const int* tokens, const int* positions, float* h, int rows, int d,
                 int vocab, int n_pos, cudaStream_t s);
// h[r,:] = src[r,:] (f32) + wpe[pos0 + r % S, :]   -- prefill of externally supplied embeddings
int add_positions(const float* src, const bf16* wpe, int pos0, int S, float* h, int rows, int d, cudaStream_t s);
// copy rows of a strided f32 block: dst[r, :] = src[(r / gi) * go + off + r % gi, :]
int gather_rows_f32(const float* src, long long lds, int gi, int go, int off, float* dst, long long ldd, int rows,
                    int d, cudaStream_t s);

// weight ingestion: cast (and transpose) caller tensors of dtype {0 f32, 1 f16, 2 bf16} into library storage
int convert_rows_bf16(const void* src, int dtype, long long rows, int cols, bf16* dst, long long dst_ld,
                      cudaStream_t s);
int convert_f32(const void* src, int dtype, long long n, float* dst, cudaStream_t s);
int transpose_bf16(const void* src, int dtype, int R, int C, bf16* dst /*[C, R]*/, long long dst_ld, cudaStream_t s);

// ------------------------------------------------------------------ image preprocessing (preprocess.cu)
size_t preprocess_scratch_bytes(int H, int W, int new_h, int new_w, int n_px);
int preprocess_image(const uint8_t* rgb, int H, int W, int new_h, int new_w, int top, int left, int n_px, const float* mean,
                     const float* stdv, float* out, void* scratch, size_t scratch_bytes, cudaStream_t s);

// ------------------------------------------------------------------ attention (attention.cu)
struct KvCache {
  bf16* base = nullptr;     // [L][2][num_pages][H][page_tokens][hd]
  int L = 0, H = 0, hd = 0, page_tokens = 0, num_pages = 0;
  int max_pages_per_row = 0;
  size_t layer_stride() const { return 2ull * num_pages * H * page_tokens * hd; }
  size_t kv_stride() const { return 1ull * num_pages * H * page_tokens * hd; }
};
// Full attention over a sequence held in one fused qkv buffer [B*S, 3*d] (q | k | v, head h at h*hd); S > 256 only for
// non-causal attention without cache, rotary or key mask, with hd % 8 == 0 and hd <= 256 (attention_prefill_unsupported).
// causal=0: ViT / mapper; causal=1: LM prefill, which also stores K/V into cache pages through block_table
// ([B, max_pages_per_row] int32) at positions pos0..pos0+S-1 and (GPT-J) applies rotary to q/k first.
// key_mask: optional [B, S] uint8, 0 = key may not be attended (HF attention_mask).
int attention_prefill(const bf16* qkv, bf16* out, int B, int S, int H, int hd, float scale, int causal,
                      const KvCache* cache, int layer, const int* block_table, int pos0, int rotary_dim,
                      const uint8_t* key_mask, cudaStream_t s);
// nullptr when attention_prefill has a kernel for the shape, else why not.  attention_prefill rejects exactly these shapes
// (cudaErrorInvalidValue); ccb_create and the LM entry points call it up front so that a shape no kernel holds fails with
// this reason before anything is launched.  Above 256 tokens see attention_prefill_long; at most 256 the scalar kernel
// takes what mma.sync / tcgen05 do not, as long as K and V of the sequence fit its 200 KB of shared memory
// (S * (4 * hd + 36) + 32 * hd + 4 bytes: GPT-J's head_dim 256 up to S = 185, head_dim 200 up to 237, 512 up to 90).
const char* attention_prefill_unsupported(int S, int hd, int causal, bool cache, int rotary_dim, bool key_mask);
// S > 256 part of attention_prefill (attention_long.cu): non-causal, unmasked, no cache / rotary, hd % 8 == 0, hd <= 256
int attention_prefill_long(const bf16* qkv, bf16* out, int B, int S, int H, int hd, float scale, cudaStream_t s);
// One new token per row: appends this step's k/v (from qkv [B, 3*d]) at position ctx_len[b] and attends over
// positions [0, ctx_len[b]] through the block table. ctx_len is device memory (graph-replay friendly).  `out` rows have pitch ldo
// (elements): H * hd, or wider when the output lands in the [att | mlp] operand of GPT-J's fused out_proj + fc_out GEMM.
int attention_decode(const bf16* qkv, bf16* out, long long ldo, int B, int H, int hd, float scale, const KvCache* cache, int layer,
                     const int* block_table, const int* ctx_len, int rotary_dim, cudaStream_t s);

// ------------------------------------------------------------------ samplers (sampler.cu)
struct SamplerScratch {
  void* buf = nullptr;
  size_t bytes = 0;
};
// greedy: next[b] = argmax_v logits[b, v] (lowest index wins ties)
int sample_greedy(const float* logits, long long ld, int B, int V, int* next, cudaStream_t s);
// mean cross entropy over the rows whose target != ignore_index; row_loss [rows], out2 = {mean, counted rows}
int cross_entropy(const float* logits, long long ld, int rows, int V, const int* targets, const int* row_map, int ignore_index,
                  float* row_loss, float* out2, cudaStream_t s);
// nucleus / top-k sampling following sampling.py:114-162 + multinomial (== argmax(p / q), q ~ Exp(1)):
//   logits <- repetition penalty over history (optional) -> / temperature -> top-k -> top-p -> typical-p -> softmax -> sample
// top_p / top_k may be per-row device arrays (or null -> scalar). q_noise [B, ldq] f32 Exp(1) samples or null
// -> in-kernel Philox keyed by (seed, row_id[b], step).
struct SampleParams {
  float temperature = 1.f;
  float top_p = 0.f;
  int top_k = 0;
  const float* top_p_rows = nullptr;
  const int* top_k_rows = nullptr;
  float typ_p = 0.f;                   // typical decoding budget (sampling.py:72-102); <= 0 disables
  const float* typ_p_rows = nullptr;   // per-row budgets: the filter then runs on every row (reference: any(typ_p > 0))
  float repetition_penalty = 1.f;
  const int* history = nullptr;  // [B, ld_hist] tokens generated so far
  long long ld_hist = 0;
  const int* hist_len = nullptr;  // device [B] or null
  int hist_len_scalar = 0;
  int hist_len_from_step = 0;     // 1: history length = *step (tokens generated so far in the on-device loop)
  const float* q_noise = nullptr; // row b of step t at q_noise + t * q_step_stride + b * ldq
  long long ldq = 0;
  long long q_step_stride = 0;
  unsigned long long seed = 0;
  const long long* row_ids = nullptr;  // global image ids for the Philox key (null -> row index)
  const int* step = nullptr;           // device step counter (null -> step_scalar)
  int step_scalar = 0;
  float* filtered_out = nullptr;       // optional [B, ld] masked logits (for parity tests of the processors)
  int* alt_out = nullptr;              // optional second sample (multinomial(p, 2) column 1)
};
int sample_top_p(const float* logits, long long ld, int B, int V, const SampleParams& sp, int* next,
                 cudaStream_t s);
// One beam-search step for N images x beam rows (inference.py:98-131 semantics per image).
struct BeamState {
  float* scores = nullptr;       // [N, beam]
  float* seq_lengths = nullptr;  // [N, beam] (f32 like the reference)
  uint8_t* has_stopped = nullptr;  // [N, beam]
  int* tokens = nullptr;         // [N, beam, max_len]
  int max_len = 0;
  const int* step = nullptr;     // device step counter: 0 = first step (topk over the single prefill row)
  void* cand_scratch = nullptr;  // [cand_rows, kBeamCandPerRow] (value, flat index) pairs: the rows' best candidates
  int cand_rows = 0;
};
constexpr int kBeamCandPerRow = 8;   // == kMaxBeam of sampler.cu
int beam_step(const float* logits, long long ld, int N, int beam, int V, float temperature, int stop_token,
              const BeamState& st, int* next_tokens /*[N*beam]*/, int* src_rows /*[N*beam] global row ids*/,
              int* block_table /*[N*beam, max_pages] permuted in place, or null*/, int max_pages,
              const int* ctx_len /*[N*beam] cached tokens per row*/, cudaStream_t s);
// Per-step bookkeeping after a sampled token: tokens_out[r, *step] = next[r]; stop counting (stop_token up to
// max_stops, eos_token) -> lengths / finished; *step += 1.  Null pointers skip the corresponding part.
int advance_rows(const int* next, int rows, int* tokens_out, int max_len, int* lengths, int* stops, uint8_t* finished,
                 int* ctx_len, int* step, int stop_token, int max_stops, int eos_token, cudaStream_t s);
// x[r] += 1 for r < rows; *scalar += 1 when non-null
int increment_rows(int* x, int rows, int* scalar, cudaStream_t s);

}  // namespace ccb
