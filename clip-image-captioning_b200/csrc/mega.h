// Persistent decode-step kernel ("mega"): one cooperative launch of one CTA per SM runs embed -> all transformer
// layers -> ln_f for up to 256 rows (one new token each) of a GPT-2 style model.  See decode_mega.cu.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <vector>

#include "internal.h"

namespace ccb {

struct MegaLayer {  // device pointers of one layer's vectors (f32)
  const float *ln1_g, *ln1_b, *ln2_g, *ln2_b;
  const float *b_qkv, *b_proj, *b_fc, *b_fc2;
};

// One of the four weight matrices of a layer, [rows_out, 64 * kb] K-major, cut into units of 128 rows x 64 k.
// The units of a matrix (row-tile major, then k) are dealt to the CTAs in equal contiguous ranges ("stream-K"):
// CTA c owns units [c * units / ncta, (c + 1) * units / ncta).  A row tile is therefore summed by a few CTAs; CTA c
// writes its fp32 partial of tile t to slot (c - first_cta(t)) of the workspace and the consumer phase adds the
// nslots(t) slots in slot order (deterministic, no atomics).
struct MegaGemmShape {
  int rows_out, kb, tiles, units, tbl_off;
};

struct MegaParams {
  int L, d, H, ff, R, N, ncta;
  float eps, scale;
  const MegaLayer* layers;     // [L]
  const CUtensorMap* wmaps;    // [L * 4] device array: qkv, proj, fc, fc2; box {64, 128}, 128B swizzle
  const uint32_t* tile_tbl;    // per gemm kind, per row tile: first_cta | nslots << 16
  int tbl_entries;
  MegaGemmShape g[4];
  float* h;                    // [R, d] residual stream
  bf16* x;                     // [R, d] LayerNorm output (operand of qkv and fc); ln_f output at exit
  bf16* att;                   // [R, d]
  bf16* mlp;                   // [R, ff]
  float* ws;                   // split-K partials [slot][R][rows_out]
  const bf16* wte;
  const bf16* wpe;
  const int* tokens;           // [R] token to embed
  const int* ctx_len;          // [R] cached tokens per row == position of the new token
  const int* block_table;
  KvCache kv;
  const float *lnf_g, *lnf_b;
  unsigned int* sync;          // [0] phase counter (zero at entry and at exit)
  int nW, nX, sc_cap;          // ring depths, per-warp score capacity (floats)
  int grp;                     // units per ring hand-over (2: slot pairs, 1: single slots)
  int log2_page_tokens;
  int xring_bytes;             // X ring size (>= 64 KB: it doubles as the scratch of the vector phases)
  int nbar;                    // grid barriers per launch minus the exit barrier (8 * L): sizes the trace rows
  unsigned long long* trace;   // optional [ncta][2 * (8 * L + 1)] globaltimer stamps of CTA phases
};

// host-side plan, owned by ccb_ctx
struct MegaState {
  bool available = false;      // model shape supported and buffers allocated
  bool enabled = false;        // CCB_MEGA=0 in the environment or ccb_debug_set_mega(ctx, 0) switches it off
  int ncta = 0;
  int max_rows = 0;            // rows the workspace was sized for (<= 256)
  MegaGemmShape g[4] = {};
  int tbl_entries = 0;
  CUtensorMap* d_wmaps = nullptr;
  MegaLayer* d_layers = nullptr;
  uint32_t* d_tbl = nullptr;
  float* d_ws = nullptr;
  unsigned int* d_sync = nullptr;
  unsigned long long* trace = nullptr;
  std::vector<uint32_t> h_tbl;
  size_t ws_floats_per_row = 0;
};

// fills g[] / table for `ncta` CTAs; returns max over kinds of (max slots * rows_out) = workspace floats per row
size_t mega_plan(MegaState& m, int d, int ff, int ncta);

// 2-D bf16 [rows, K] tensor map with box {64, box_rows} and the 128B swizzle (gemm.cu)
int gemm_make_tmap(CUtensorMap* m, const void* ptr, uint64_t rows, uint64_t K, uint64_t ld, uint32_t box_rows);

// launches the kernel (cooperative); returns 0 / cudaError / -1 (gemm_last_error)
int mega_launch(const MegaParams& p, cudaStream_t s);
int mega_init();  // function attributes

}  // namespace ccb
