// bf16 x bf16 -> fp32 GEMM for sm_100a, one output tile per CTA: TMA (128B-swizzled K-major tiles) -> tcgen05.mma with
// the accumulator in TMEM -> tcgen05.ld epilogue with fused bias / activation / residual and a transposed store.
//
//   out[j, i] = sum_k A[i, k] * B[j, k]      A = weights [features, K], B = activations [tokens, K], bf16 row-major
//
// This is the "swapped" orientation of gemm.cu, used when tokens <= 256 (decode): the 128-row MMA tile is filled by
// weight rows and every weight byte is streamed once.  Token-heavy contractions (tokens on the 128-row side) run on the
// persistent kernels of gemm_persist.cuh.
//
// One CTA computes one 128 x BN tile (optionally one K-split of it).  Warp roles: warp 0 = TMA producer,
// warp 1 = TMEM allocator + MMA issuer (one elected lane), warps 2..5 = epilogue (one TMEM lane quadrant
// each).  Split-K (used to fill the 148 SMs when there are few output tiles, i.e. in decode) runs the S splits of
// one tile as ONE thread-block cluster (1,1,S): every CTA parks its fp32 accumulator in its own shared memory,
// the cluster synchronises, and CTA z reduces the 8-column groups c with c % S == z by reading the S partial
// tiles over distributed shared memory in the fixed order 0..S-1 (deterministic, no global workspace, no
// atomics) before running the fused epilogue on them.
#pragma once
#include "common.cuh"
#include "ptx.cuh"

namespace ccb {

struct GemmParams {
  int Ra, Rb;        // valid rows of A (features) / B (tokens): tile rows beyond are zero-filled by TMA and masked at the store
  int k_blocks;      // K / 64
  int split_k;       // >= 1; == cluster size along z
  // epilogue: out[j * ldo + i] = act(acc[i, j] + bias[i]) + residual[j * ldr + i]
  void* out;         // f32 or bf16
  int out_bf16;
  long long ldo;
  const float* bias;       // per feature i; may be null
  const float* residual;   // f32; may be null (may alias out)
  long long ldr;
  int act;
  // 1: launched with programmatic stream serialization inside the engine's chain: weight tiles are fetched
  // before the dependency wait (they are never produced by the preceding kernel)
  int pdl;
  // optional timeline for tuning: 8 globaltimer stamps per CTA (null in production)
  unsigned long long* trace;
};

template <int BN>
struct GemmCfg {
  static constexpr int BM = 128;
  static constexpr int BK = 64;
  static constexpr int kStages = (BN >= 256) ? 4 : (BN >= 128 ? 5 : 3);   // BN = 32: two CTAs per SM; BN = 64 without split-K: three
  static constexpr int kMinBlocks = 1;
  static constexpr int kABytes = BM * BK * 2;
  static constexpr int kBBytes = BN * BK * 2;
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kTmemCols = BN < 32 ? 32 : BN;
  // Split-K staging (see the kernel): S slots x ceil(BN/8 / S) column groups x 8 columns x 128 rows of f32 per
  // CTA, at most (BN/8 + 8) groups of 4 KB.  Decode tiles (BN <= 64) get their own region so that peers may push
  // into it while this CTA's pipeline is still running (one cluster barrier); larger tiles reuse the pipeline
  // stages after an extra barrier.
  static constexpr bool kSeparateStaging = (BN <= 64);
  static constexpr int kStagingBytes = (BN / 8 + 8) * 4096;
  static_assert(kSeparateStaging || kStages * kStageBytes >= kStagingBytes, "staging must fit in the pipeline buffers");
  static constexpr int kSmemBytes = kStages * kStageBytes + (kSeparateStaging ? kStagingBytes : 0) + 1024 /*align slack*/ +
                                    256 /*barriers*/;
  static constexpr int kThreads = 192;
};

// per-CTA timeline stamps: compiled in only with -DCCB_TUNING (python tools/build.py --tuning)
#ifdef CCB_TUNING
#define CCB_TRACE(slot)                                                                                   \
  do {                                                                                                    \
    if (p.trace != nullptr && lane == 0)                                                                  \
      p.trace[((blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x) * 8ull + (slot)] = ptx::globaltimer_ns(); \
  } while (0)
#else
#define CCB_TRACE(slot) do { } while (0)
#endif

// The fused epilogues (gemm_epilogue_transposed below, persist_epilogue_cols in gemm_persist.cuh) are kept small on
// purpose: they run once per tile, so their instructions are cold in the instruction cache (a fully unrolled epilogue
// with the activation switch inlined was 22 K instructions and cost ~15 us per tile in instruction fetches).
template <int CW>
__device__ __forceinline__ void gemm_apply_act(float (&acc)[CW], int act) {
  if (act == ACT_RELU) {
#pragma unroll
    for (int v = 0; v < CW; ++v) acc[v] = fmaxf(acc[v], 0.f);
  } else if (act == ACT_GELU_NEW) {
    // 0.5 x (1 + tanh(u)) == x - x / (1 + exp(2u)); exp2-based __expf + fast divide: ~1e-6 relative error, far
    // below the bf16 rounding of the stored value, and a handful of instructions (the epilogue has 4 warps)
#pragma unroll
    for (int v = 0; v < CW; ++v) {
      const float x = acc[v];
      const float u = 0.7978845608028654f * (x + 0.044715f * x * x * x);
      acc[v] = x - __fdividef(x, 1.f + __expf(2.f * u));
    }
  } else if (act == ACT_QUICKGELU) {
#pragma unroll
    for (int v = 0; v < CW; ++v) acc[v] = __fdividef(acc[v], 1.f + __expf(-1.702f * acc[v]));
  } else if (act != ACT_NONE) {
#pragma unroll
    for (int v = 0; v < CW; ++v) acc[v] = apply_act_call(acc[v], act);  // static indices keep acc in registers
  }
}

// Epilogue of feature i (this thread's accumulator row) for the 8 tokens [j0, j0 + 8).
__device__ __forceinline__ void gemm_epilogue_transposed(const GemmParams& p, float (&acc)[8], int i, bool i_ok,
                                                         float bias_i, int j0) {
  if (!i_ok) return;
#pragma unroll
  for (int v = 0; v < 8; ++v) acc[v] += bias_i;
  gemm_apply_act(acc, p.act);
  // lanes hold consecutive features i -> coalesced accesses for every token j.  All residual loads are issued
  // before the first store: out may alias residual (in-place residual stream), so a load placed after a store
  // could not be hoisted by the compiler and the 8 load latencies would serialise.
  if (p.residual) {
    float res[8];
#pragma unroll
    for (int v = 0; v < 8; ++v) res[v] = (j0 + v < p.Rb) ? p.residual[static_cast<long long>(j0 + v) * p.ldr + i] : 0.f;
#pragma unroll
    for (int v = 0; v < 8; ++v) acc[v] += res[v];
  }
#pragma unroll
  for (int v = 0; v < 8; ++v) {
    const int j = j0 + v;
    if (j < p.Rb) {
      if (p.out_bf16)
        reinterpret_cast<__nv_bfloat16*>(p.out)[static_cast<long long>(j) * p.ldo + i] = __float2bfloat16_rn(acc[v]);
      else
        reinterpret_cast<float*>(p.out)[static_cast<long long>(j) * p.ldo + i] = acc[v];
    }
  }
}

template <int BN>
__global__ void __launch_bounds__(192, GemmCfg<BN>::kMinBlocks) gemm_bf16_tn_kernel(const __grid_constant__ CUtensorMap tma_a,
                                                           const __grid_constant__ CUtensorMap tma_b,
                                                           const GemmParams p) {
  using Cfg = GemmCfg<BN>;
  constexpr int kStages = Cfg::kStages;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (ptx::smem_u32(smem_raw) + 1023u) & ~1023u;
  // (the separate split-K staging area exists only in split-K launches: see the launcher)
  const uint32_t kDataBytes = kStages * Cfg::kStageBytes + ((Cfg::kSeparateStaging && p.split_k > 1) ? Cfg::kStagingBytes : 0);
  const uint32_t bar_base = smem_base + kDataBytes;
  // barrier layout: full[kStages], empty[kStages], tmem_full, then the TMEM address slot
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (kStages + s); };
  const uint32_t tmem_full_bar = bar_base + 8u * (2 * kStages);
  const uint32_t tmem_slot = bar_base + 8u * (2 * kStages + 1);
  uint8_t* smem_gen = smem_raw + (smem_base - ptx::smem_u32(smem_raw));
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_gen + kDataBytes + 8 * (2 * kStages + 1));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  if (warp == 0) CCB_TRACE(0);  // entry

  // K range of this split (blockIdx.z == rank in the cluster)
  const int kb_per = (p.k_blocks + p.split_k - 1) / p.split_k;
  const int kb_begin = blockIdx.z * kb_per;
  int kb_end = kb_begin + kb_per;
  if (kb_end > p.k_blocks) kb_end = p.k_blocks;
  const int nkb = kb_end - kb_begin;  // host guarantees >= 1 for every split

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tma_a);
    ptx::prefetch_tmap(&tma_b);
    for (int s = 0; s < kStages; ++s) {
      ptx::mbar_init(full_bar(s), 1);
      ptx::mbar_init(empty_bar(s), 1);
    }
    ptx::mbar_init(tmem_full_bar, 1);
    ptx::fence_mbar_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc<Cfg::kTmemCols>(tmem_slot);
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;
  if (warp == 0) CCB_TRACE(1);  // setup done
  ptx::grid_dep_launch();       // the next kernel of the stream may start its prologue now
  if (p.split_k > 1) ptx::cluster_arrive();  // "this CTA is running": completed by the wait ahead of the pushes

  const int row_a0 = blockIdx.x * Cfg::BM;
  const int row_b0 = blockIdx.y * BN;
  const int quad = warp & 3;  // TMEM lane quadrant an epilogue warp may access
  const int i = row_a0 + quad * 32 + lane;
  const bool i_ok = i < p.Ra;
  const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quad * 32) << 16);
  const uint32_t red_base = smem_base + (Cfg::kSeparateStaging ? kStages * Cfg::kStageBytes : 0);  // split-K staging

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    if (lane == 0) {
      // weights (A) are streamed once (evict-first); activations (B) are re-read by many CTAs (evict-last).  The weights
      // do not depend on the preceding kernel: with PDL their first kStages tiles are requested before the dependency
      // wait, the activation tiles right after it.
      const int pre = p.pdl ? (nkb < kStages ? nkb : kStages) : 0;
      for (int it = 0; it < pre; ++it) {
        ptx::mbar_arrive_expect_tx(full_bar(it), Cfg::kStageBytes);
        ptx::tma_load_2d(smem_base + it * Cfg::kStageBytes, &tma_a, full_bar(it), (kb_begin + it) * Cfg::BK, row_a0, ptx::kEvictFirst);
      }
      ptx::grid_dep_wait();
      for (int it = 0; it < pre; ++it)
        ptx::tma_load_2d(smem_base + it * Cfg::kStageBytes + Cfg::kABytes, &tma_b, full_bar(it), (kb_begin + it) * Cfg::BK, row_b0,
                         ptx::kEvictLast);
      for (int it = pre; it < nkb; ++it) {
        const int s = it % kStages;
        const uint32_t ph = (it / kStages) & 1;
        ptx::mbar_wait(empty_bar(s), ph ^ 1);
        const uint32_t st = smem_base + s * Cfg::kStageBytes;
        ptx::mbar_arrive_expect_tx(full_bar(s), Cfg::kStageBytes);
        const int kcoord = (kb_begin + it) * Cfg::BK;
        ptx::tma_load_2d(st, &tma_a, full_bar(s), kcoord, row_a0, ptx::kEvictFirst);
        ptx::tma_load_2d(st + Cfg::kABytes, &tma_b, full_bar(s), kcoord, row_b0, ptx::kEvictLast);
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer
    if (lane == 0) {
      constexpr uint32_t idesc = ptx::umma_idesc_bf16(Cfg::BM, BN);
      for (int it = 0; it < nkb; ++it) {
        const int s = it % kStages;
        const uint32_t ph = (it / kStages) & 1;
        ptx::mbar_wait(full_bar(s), ph);
        ptx::tc_fence_after();
        if (it == 0) CCB_TRACE(2);  // first stage landed
        const uint32_t sa = smem_base + s * Cfg::kStageBytes;
        const uint32_t sb = sa + Cfg::kABytes;
        const uint64_t adesc = ptx::umma_desc_k_sw128(sa);
        const uint64_t bdesc = ptx::umma_desc_k_sw128(sb);
#pragma unroll
        for (int k = 0; k < Cfg::BK / 16; ++k) {
          // advance 16 bf16 = 32 bytes along K inside the 128B swizzle atom: +2 in the (addr>>4) field
          ptx::umma_bf16(tmem_base, adesc + 2u * k, bdesc + 2u * k, idesc, (it > 0 || k > 0) ? 1u : 0u);
        }
        ptx::umma_commit(empty_bar(s));  // frees the smem stage when these MMAs retire
      }
      ptx::umma_commit(tmem_full_bar);   // accumulator complete
      CCB_TRACE(3);                      // all MMAs issued
    }
    __syncwarp();
  } else {
    // ------------------------------------------------------------ epilogue warps 2..5: accumulator is ready
    ptx::grid_dep_wait();  // (returns at once unless this is a PDL launch) before any global read / write below
    ptx::mbar_wait(tmem_full_bar, 0);
    ptx::tc_fence_after();
    if (warp == 2) CCB_TRACE(4);  // accumulator ready
  }

  if (p.split_k > 1) {
    // ------------------------------------------------------------ split-K: push-based cluster reduction
    // The BN/8 groups of 8 columns are dealt round-robin to the S CTAs of the cluster (owner of group c = c % S).
    // Every CTA PUSHES its partial of group c into slot [its rank] of the owner's staging area with fire-and-forget
    // remote stores (no load round trips over the cluster network); after one cluster barrier each owner sums
    // its slots in the fixed order 0..S-1 (deterministic) out of its OWN shared memory and runs the epilogue.
    const uint32_t S = p.split_k;
    const uint32_t my_rank = blockIdx.z;
    const uint32_t NC = BN / 8;
    const uint32_t MPO = (NC + S - 1) / S;  // groups per owner (upper bound)
    ptx::cluster_wait();          // every CTA of the cluster has started: its shared memory may be written
    if (!Cfg::kSeparateStaging) {
      // the staging area aliases the pipeline stages: peers may only write once every CTA's MMAs have retired
      ptx::cluster_arrive();
      ptx::cluster_wait();
    }
    if (warp >= 2) {
      const uint32_t row_off = static_cast<uint32_t>(quad * 32 + lane) * 4u;
#pragma unroll 1
      for (uint32_t c = 0; c < NC; ++c) {
        uint32_t r[8];
        ptx::tmem_ld8(taddr + c * 8, r);
        ptx::tmem_ld_wait();
        const uint32_t local = red_base + ((my_rank * MPO + c / S) * 8u) * 512u + row_off;
        const uint32_t remote = ptx::mapa_shared(local, c % S);
#pragma unroll
        for (int v = 0; v < 8; ++v) ptx::st_dsmem_f32(remote + v * 512u, __uint_as_float(r[v]));
      }
    }
    ptx::cluster_arrive();        // release: the pushes above are visible to the owners after the wait
    ptx::cluster_wait();
    if (warp == 2) CCB_TRACE(5);
    if (warp >= 2) {
      const float bias_i = (p.bias != nullptr && i_ok) ? p.bias[i] : 0.f;
      const uint32_t row_off = static_cast<uint32_t>(quad * 32 + lane) * 4u;
#pragma unroll 1
      for (uint32_t c = my_rank, li = 0; c < NC; c += S, ++li) {
        const int j0 = row_b0 + static_cast<int>(c) * 8;
        if (j0 >= p.Rb) break;
        float acc[8];
#pragma unroll
        for (int v = 0; v < 8; ++v) acc[v] = 0.f;
#pragma unroll 1
        for (uint32_t sl = 0; sl < S; ++sl) {        // fixed order 0..S-1: deterministic sum
          const uint32_t src = red_base + ((sl * MPO + li) * 8u) * 512u + row_off;
#pragma unroll
          for (int v = 0; v < 8; ++v) acc[v] += ptx::ld_shared_f32(src + v * 512u);
        }
        gemm_epilogue_transposed(p, acc, i, i_ok, bias_i, j0);
      }
      if (warp == 2) CCB_TRACE(6);  // epilogue done
    }
  } else if (warp >= 2) {
    const float bias_i = (p.bias != nullptr && i_ok) ? p.bias[i] : 0.f;
#pragma unroll 1
    for (int c0 = 0; c0 < BN; c0 += 8) {
      const int j0 = row_b0 + c0;
      if (j0 >= p.Rb) break;
      uint32_t r[8];
      ptx::tmem_ld8(taddr + c0, r);
      ptx::tmem_ld_wait();
      float acc[8];
#pragma unroll
      for (int v = 0; v < 8; ++v) acc[v] = __uint_as_float(r[v]);
      gemm_epilogue_transposed(p, acc, i, i_ok, bias_i, j0);
    }
    if (warp == 2) CCB_TRACE(6);  // epilogue done
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc<Cfg::kTmemCols>(tmem_base);
  }
  if (warp == 0) CCB_TRACE(7);  // exit
}

}  // namespace ccb
