// Host side of the tcgen05 GEMM: tensor-map encoding, orientation / tile / split-K selection, launch.
#include <cuda.h>
#include <stdio.h>
#include <string.h>

#include <mutex>

#include "gemm_persist.cuh"
#include "gemm_sm100.cuh"
#include "internal.h"
#include "mega.h"

namespace ccb {

namespace {

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn g_encode = nullptr;
char g_err[512] = {0};
int g_attr_status = 0;

int fail(const char* fmt, const char* detail = "") {
  snprintf(g_err, sizeof(g_err), fmt, detail);
  return -1;
}

// 2-D bf16 tensor [rows, K] with row pitch `ld` elements; box = {64 (K), box_rows}; 128B swizzle.
int make_tmap(CUtensorMap* m, const void* ptr, uint64_t rows, uint64_t K, uint64_t ld, uint32_t box_rows) {
  if ((reinterpret_cast<uintptr_t>(ptr) & 15) != 0) return fail("GEMM operand not 16-byte aligned");
  if ((ld * 2) % 16 != 0) return fail("GEMM operand row pitch not a multiple of 16 bytes");
  cuuint64_t dims[2] = {K, rows};
  cuuint64_t strides[1] = {ld * 2};
  cuuint32_t box[2] = {64, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = g_encode(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    char b[64];
    snprintf(b, sizeof(b), "%d", static_cast<int>(r));
    return fail("cuTensorMapEncodeTiled failed (CUresult %s)", b);
  }
  return 0;
}

template <int BN>
int set_attr() {
  cudaError_t e = cudaFuncSetAttribute(gemm_bf16_tn_kernel<BN>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       GemmCfg<BN>::kSmemBytes);
  if (e != cudaSuccess) return fail("cudaFuncSetAttribute(smem) failed: %s", cudaGetErrorString(e));
  return 0;
}

template <int BN>
int launch(const CUtensorMap& ta, const CUtensorMap& tb, const GemmParams& p, dim3 grid, cudaStream_t s) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid;
  cfg.blockDim = dim3(GemmCfg<BN>::kThreads);
  // without split-K the staging area of the cluster reduction is not touched: leaving it out lets several CTAs share an
  // SM (BN = 64, three stages: 74 KB instead of 138 KB, three CTAs per SM), e.g. the 393 tiles of the GPT-2 lm_head run
  // in one wave instead of 2.7
  cfg.dynamicSmemBytes = (p.split_k == 1 && GemmCfg<BN>::kSeparateStaging) ? GemmCfg<BN>::kSmemBytes - GemmCfg<BN>::kStagingBytes
                                                                         : GemmCfg<BN>::kSmemBytes;
  cfg.stream = s;
  cudaLaunchAttribute attr[2];
  int na = 0;
  if (p.split_k > 1) {
    // the S splits of one output tile form one cluster and reduce over distributed shared memory
    attr[na].id = cudaLaunchAttributeClusterDimension;
    attr[na].val.clusterDim.x = 1;
    attr[na].val.clusterDim.y = 1;
    attr[na].val.clusterDim.z = static_cast<unsigned>(p.split_k);
    ++na;
  }
  if (p.pdl) {
    attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[na].val.programmaticStreamSerializationAllowed = 1;
    ++na;
  }
  cfg.attrs = attr;
  cfg.numAttrs = na;
  cudaError_t e = cudaLaunchKernelEx(&cfg, gemm_bf16_tn_kernel<BN>, ta, tb, p);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return fail("GEMM launch failed: %s", cudaGetErrorString(e));
  }
  return 0;
}


// Kernel variant and tile width BN for the persistent kernels, from the B200 sweeps of tools/sweep_gemm_bn.py.
//  * single CTA (128-token tiles): a round of tiles costs k_blocks x the time of one k-block, which is bound by the
//    SM's shared-memory port (TMA writes and MMA reads of 16 KB + BN x 128 B each), i.e. proportional to 16 + BN / 8,
//    plus a small hand-over; rounds = ceil(tiles / SMs); the widest candidate wins ties.
//  * CTA pair (256-token tiles, half the W bytes per SM): a round costs ~max(26, 3 BN / 16) in the same units (MMA
//    bound, with a floor), rounds = ceil(tiles / pairs); it is ahead once the problem runs three or more rounds of
//    long-enough tiles (K >= 1280) or K is very long, and behind on one- or two-round problems (cluster launch and
//    synchronisation, no overlap to win back).
void pick_persist(int tokens, int features, int k_blocks, int num_sms, int force_orientation, int force_bn, bool* pair_out,
                  int* bn_out) {
  const int m_tiles = (tokens + 127) / 128;
  long long best = 0, best_rounds = 0;
  int best_bn = 0;
  for (int bn = 256; bn >= (force_bn ? 32 : 64); bn -= 32) {
    if (force_bn && bn != force_bn) continue;
    const long long tiles = static_cast<long long>(m_tiles) * ((features + bn - 1) / bn);
    const long long rounds = (tiles + num_sms - 1) / num_sms;
    const long long cost = rounds * (16 + bn / 8 + 2);
    if (best_bn == 0 || cost < best) {
      best = cost;
      best_bn = bn;
      best_rounds = rounds;
    }
  }
  bool pair = force_orientation == 3;
  if (force_orientation != 3 && force_orientation != 4)
    pair = tokens >= 512 && (k_blocks >= 64 || (best_rounds >= 3 && k_blocks >= 20));
  if (pair && !force_bn) {
    const int m2 = (tokens + 255) / 256, pairs = num_sms / 2;
    long long pbest = 0;
    for (int bn = 256; bn >= 64; bn -= 32) {
      const long long tiles = static_cast<long long>(m2) * ((features + bn - 1) / bn);
      const long long rounds = (tiles + pairs - 1) / pairs;
      const long long per = 3 * bn / 16 > 26 ? 3 * bn / 16 : 26;
      const long long cost = rounds * per * 64 + bn;   // (+ bn: the narrower tile wins ties)
      if (bn == 256 || cost < pbest) {
        pbest = cost;
        best_bn = bn;
      }
    }
  }
  *bn_out = best_bn ? best_bn : force_bn;
  *pair_out = pair;
}

int launch_persist(const GemmArgs& a, int bn, bool pair, int pdl, int num_sms, cudaStream_t s) {
  PersistParams pp;
  memset(&pp, 0, sizeof(pp));
  pp.tokens = a.tokens;
  pp.features = a.features;
  pp.k_blocks = a.K / 64;
  pp.out = a.out;
  pp.out_bf16 = a.out_bf16;
  pp.ldo = a.ldo;
  pp.bias = a.bias;
  pp.residual = a.residual;
  pp.ldr = a.ldr;
  pp.act = a.act_fn;
  pp.rg_in = a.rg_in;
  pp.rg_out = a.rg_out;
  pp.rg_off = a.rg_off;
  pp.bn = bn;
  const int stage_bytes = 128 * 128 + bn * (pair ? 64 : 128);
  int stages = (kPersistSmemBytes - 1024 - 512) / stage_bytes;
  if (stages > 8) stages = 8;
  pp.stages = stages;
  pp.m_tiles = pair ? (a.tokens + 255) / 256 : (a.tokens + 127) / 128;
  pp.n_tiles = (a.features + bn - 1) / bn;
  CUtensorMap tx, tw;
  if (make_tmap(&tx, a.act, a.tokens, a.K, a.lda, 128)) return -1;
  if (make_tmap(&tw, a.weight, a.features, a.K, a.ldw ? a.ldw : a.K, pair ? bn / 2 : bn)) return -1;
  const int tiles = pp.m_tiles * pp.n_tiles;
  const int units = pair ? num_sms / 2 : num_sms;
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3((tiles < units ? tiles : units) * (pair ? 2 : 1));
  cfg.blockDim = dim3(kPersistThreads);
  cfg.dynamicSmemBytes = static_cast<size_t>(stages) * stage_bytes + 1024 + 512;
  cfg.stream = s;
  cudaLaunchAttribute attr[2];
  int na = 0;
  if (pair) {
    attr[na].id = cudaLaunchAttributeClusterDimension;
    attr[na].val.clusterDim.x = 2;
    attr[na].val.clusterDim.y = 1;
    attr[na].val.clusterDim.z = 1;
    ++na;
  }
  if (pdl) {
    attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[na].val.programmaticStreamSerializationAllowed = 1;
    ++na;
  }
  cfg.attrs = attr;
  cfg.numAttrs = na;
  cudaError_t e = pair ? cudaLaunchKernelEx(&cfg, gemm_pair_kernel, tx, tw, pp) : cudaLaunchKernelEx(&cfg, gemm_persist_kernel, tx, tw, pp);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return fail("persistent GEMM launch failed: %s", cudaGetErrorString(e));
  }
  return 0;
}

}  // namespace

const char* gemm_last_error() { return g_err; }

int gemm_make_tmap(CUtensorMap* m, const void* ptr, uint64_t rows, uint64_t K, uint64_t ld, uint32_t box_rows) {
  if (!g_encode) return fail("gemm_init() was not called");
  return make_tmap(m, ptr, rows, K, ld, box_rows);
}

int gemm_init(int device) {
  (void)device;
  if (!g_encode) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q);
    if (e != cudaSuccess || fn == nullptr || q != cudaDriverEntryPointSuccess)
      return fail("cuTensorMapEncodeTiled not available from the driver: %s", cudaGetErrorString(e));
    g_encode = reinterpret_cast<EncodeTiledFn>(fn);
  }
  // function attributes are per device: once per device of this process (gemm_init runs under ccb_create's device)
  static std::mutex mu;
  static int status_dev[kMaxDevices];
  static bool done_dev[kMaxDevices] = {};
  std::lock_guard<std::mutex> lock(mu);
  const int slot = current_device_slot();
  if (!done_dev[slot]) {
    int r = 0;
    r |= set_attr<32>();
    r |= set_attr<64>();
    r |= set_attr<128>();
    r |= set_attr<256>();
    if (cudaFuncSetAttribute(gemm_persist_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kPersistSmemBytes) != cudaSuccess ||
        cudaFuncSetAttribute(gemm_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kPersistSmemBytes) != cudaSuccess)
      r |= fail("cudaFuncSetAttribute(smem) failed for the persistent GEMM");
    status_dev[slot] = r;
    done_dev[slot] = true;
  }
  return status_dev[slot];
}

int gemm_launch(const GemmArgs& a, const GemmWorkspace& w, cudaStream_t stream) {
  if (!g_encode) return fail("gemm_init() was not called");
  if (a.K <= 0 || a.K % 64 != 0) return fail("GEMM K must be a positive multiple of 64");
  if (a.tokens <= 0 || a.features <= 0) return fail("GEMM with empty extent");
  // the epilogue knows activations 0..7 only (GEGLU is a separate kernel on the GEMM's output); an unknown code would
  // silently run as the identity
  if (a.act_fn < ACT_NONE || a.act_fn > ACT_TANH) {
    snprintf(g_err, sizeof(g_err), "GEMM activation %d is not an epilogue activation (0..7)", a.act_fn);
    return -1;
  }
  // pitches shorter than a row would make rows overlap: a tile would read its neighbour's K range or two rows would be
  // written to the same elements.  A remap must keep the groups' rows apart: rg_off + rg_in <= rg_out.
  if (a.lda < a.K || (a.ldw != 0 && a.ldw < a.K) || a.ldo < a.features || (a.residual && a.ldr < a.features) ||
      ((a.rg_in | a.rg_out | a.rg_off) != 0 && (a.rg_in <= 0 || a.rg_off < 0 || a.rg_off + a.rg_in > a.rg_out))) {
    snprintf(g_err, sizeof(g_err),
             "GEMM pitches out of range: K=%d features=%d lda=%lld ldw=%lld ldo=%lld ldr=%lld, remap rg_in=%d rg_out=%d "
             "rg_off=%d (need lda >= K, ldw 0 or >= K, ldo >= features, ldr >= features with a residual, and for a remap "
             "rg_in > 0, rg_off >= 0, rg_off + rg_in <= rg_out)",
             a.K, a.features, a.lda, a.ldw, a.ldo, a.ldr, a.rg_in, a.rg_out, a.rg_off);
    return -1;
  }

  // force_orientation: 0 auto, 1 normal, 2 swapped, 3 normal + CTA-pair persistent kernel, 4 normal + single-CTA persistent
  const bool swapped = a.force_orientation ? (a.force_orientation == 2) : (a.tokens <= 256);
  if (swapped && a.rg_in > 0) return fail("row remap is only supported in the normal orientation");
  if (swapped && a.tokens > 256) return fail("swapped orientation needs tokens <= 256");
  if (!swapped && a.force_split) return fail("split-K is only available in the swapped orientation");
  // tuning timelines: every launch takes the next slot, although only the one-tile kernel writes stamps
  unsigned long long* trace = w.trace ? w.trace + (w.trace_count++ % w.trace_launches) * w.trace_stride : nullptr;
  const int pdl = (a.allow_pdl && pdl_enabled()) ? 1 : 0;

  if (!swapped) {
    // token-heavy contractions (ViT / mapper / prefill) take the persistent kernels.  Their vector store path assumes
    // 16-byte aligned bases; it falls back to scalar stores through odd ldo otherwise.
    if ((reinterpret_cast<uintptr_t>(a.out) & 15) || (a.residual && (reinterpret_cast<uintptr_t>(a.residual) & 15)) ||
        (a.bias && (reinterpret_cast<uintptr_t>(a.bias) & 15)))
      return fail("normal-orientation GEMM needs 16-byte aligned out / residual / bias");
    bool pair = false;
    int bn = 0;
    pick_persist(a.tokens, a.features, a.K / 64, w.num_sms, a.force_orientation, a.force_bn, &pair, &bn);
    if (bn < 32 || bn > 256 || bn % 32) return fail("unsupported BN for the persistent GEMM");
    return launch_persist(a, bn, pair, pdl, w.num_sms, stream);
  }

  // swapped: weights on the 128-row side of the one-tile-per-CTA kernel, the tokens fill a BN-wide tile
  const int bn = a.force_bn ? a.force_bn : a.tokens <= 32 ? 32 : a.tokens <= 64 ? 64 : a.tokens <= 128 ? 128 : 256;
  if (bn != 32 && bn != 64 && bn != 128 && bn != 256) return fail("unsupported BN");
  if (bn < a.tokens) return fail("swapped orientation: BN smaller than token count");

  GemmParams p;
  memset(&p, 0, sizeof(p));
  p.Ra = a.features;
  p.Rb = a.tokens;
  p.k_blocks = a.K / 64;
  p.out = a.out;
  p.out_bf16 = a.out_bf16;
  p.ldo = a.ldo;
  p.bias = a.bias;
  p.residual = a.residual;
  p.ldr = a.ldr;
  p.act = a.act_fn;
  p.trace = trace;
  p.pdl = pdl;

  dim3 grid((p.Ra + 127) / 128, (p.Rb + bn - 1) / bn, 1);
  const int tiles = grid.x * grid.y;
  int split = 1;
  if (a.force_split) {
    split = a.force_split;
  } else {
    // fill the machine without spilling into a second wave: tiles * split <= CTA slots, each split >= 4 k-blocks.
    // A 32-token tile (3 stages of 20 KB + 48 KB of split-K staging = 109 KB) fits twice on an SM, so the decode GEMMs
    // of a 16-row GPT-J step run e.g. 96 qkv tiles x 3 splits or 32 out_proj tiles x 8 splits in one wave.
    const int slots = w.num_sms * (bn == 32 ? 2 : 1);
    if (tiles < slots) {
      split = slots / tiles;
      const int max_by_k = p.k_blocks / 4 > 0 ? p.k_blocks / 4 : 1;
      if (split > max_by_k) split = max_by_k;
      // with two CTAs per SM, clusters of 3, 5, 6 or 7 CTAs place badly on the GPCs (the 96-tile x 3 q/k/v GEMM of a 16-row
      // GPT-J step: 32 us against 26 us with pairs; GPT-J step 3.02 -> 2.91 ms): round the split down to a power of two.
      // One CTA per SM (64-token tiles: the GPT2-XL operator chain) is 2 % faster with the odd splits, so it keeps them.
      if (bn == 32)
        while (split & (split - 1)) --split;
    }
  }
  if (split > p.k_blocks) split = p.k_blocks;
  if (split > 8) split = 8;  // portable cluster size
  // every split must own at least one k-block: ceil(kb/split)*(split-1) < kb
  while (split > 1 && ((p.k_blocks + split - 1) / split) * (split - 1) >= p.k_blocks) --split;
  p.split_k = split;
  grid.z = split;

  CUtensorMap ta, tb;
  if (make_tmap(&ta, a.weight, a.features, a.K, a.ldw ? a.ldw : a.K, 128)) return -1;
  if (make_tmap(&tb, a.act, a.tokens, a.K, a.lda, bn)) return -1;

  switch (bn) {
    case 32: return launch<32>(ta, tb, p, grid, stream);
    case 64: return launch<64>(ta, tb, p, grid, stream);
    case 128: return launch<128>(ta, tb, p, grid, stream);
    default: return launch<256>(ta, tb, p, grid, stream);
  }
}

}  // namespace ccb
