// Persistent decode-step kernel for GPT-2 style models (lms/GPT2.py:17-19 -> HF GPT2LMHeadModel, one new token per
// row against the KV cache): embed -> L x [ln_1, c_attn, attention, c_proj, ln_2, c_fc, gelu_new, mlp.c_proj] -> ln_f
// in ONE cooperative launch of one CTA per SM.
//
// Why: a decode step is bound by streaming every weight once from HBM (3.1 GB for GPT2-XL) but consists of ~340
// dependent little operators; as separate kernels each of them pays launch, prologue, pipeline ramp and tail.  Here
// the weight stream never stops:
//   warp 0  W producer : walks this CTA's share of ALL weight tiles of ALL layers in consumption order and keeps a
//                        deep TMA ring (128 rows x 64 k, 16 KB per stage) full.  It depends on nothing but free ring
//                        slots, so it runs ahead of the math across operator and layer boundaries.
//   warp 1  X producer : TMA-loads the activation tile (all rows x 64 k) each unit needs, after the grid-wide phase
//                        counter says the producing phase is complete.
//   warp 2  MMA issuer : tcgen05.mma 128 x N x 16 (weights on the 128-row side, rows = N <= 256), fp32 accumulator
//                        in TMEM, double buffered.
//   warp 3             : TMEM allocation.
//   warps 4-11 compute : GEMM epilogue (TMEM -> fp32 split-K partials in an L2-resident workspace) and the vector
//                        phases between the GEMMs, which fold the partials: residual + bias + LayerNorm, attention
//                        over the paged KV cache (+ append of the new K/V), bias + gelu_new.
// Work split: stream-K (mega.h).  Phases are separated by a grid barrier (one monotonically increasing counter in
// global memory, red.release / ld.acquire); cross-CTA data is read with ld.global.cg or TMA (after a proxy fence).
//
// Everything in here runs on a handful of warps per SM with nothing to hide latency behind, so the loops are written
// for a short dependent-instruction chain: no integer division or 64-bit index arithmetic inside loops, ring stage /
// phase kept incrementally, phases as out-of-line functions (the kernel must stay resident in the instruction cache).
#include <cuda.h>
#include <stdio.h>
#include <string.h>

#include "common.cuh"
#include "mega.h"
#include "ptx.cuh"

namespace ccb {

namespace {

constexpr int kThreads = 384;
constexpr int kTblMax = 256;
constexpr int kLnSlots = 14;            // split-K slots a LayerNorm thread keeps in flight per column
constexpr int kAttnWarps = 11;           // the 8 compute warps + the X-producer, MMA and TMEM-allocator warps (idle then)
constexpr int kVecScratch = kAttnWarps * 8192;  // vector-phase scratch: the (idle) X ring and what follows it, 8 KB per warp
constexpr int kComputeThreads = 256;
constexpr int kComputeWarp0 = 4;
constexpr int kWStage = 128 * 64 * 2;

__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void red_release_add(unsigned* p, unsigned v) {
  asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ float4 ldcg_f4(const float* p) {
  float4 v;
  asm volatile("ld.global.cg.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
  return v;
}
__device__ __forceinline__ float2 ldcg_f2(const float* p) {
  float2 v;
  asm volatile("ld.global.cg.v2.f32 {%0,%1}, [%2];" : "=f"(v.x), "=f"(v.y) : "l"(p));
  return v;
}
__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }
// 16-byte asynchronous copy global -> shared; src_bytes == 0 writes zeros
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src, uint32_t src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ uint4 lds_u4(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
  return v;
}

// wait until the phase counter reaches `target` (bounded: a protocol bug traps instead of hanging the GPU)
__device__ __forceinline__ void poll_counter(const unsigned* ctr, unsigned target) {
  if (ld_acquire_u32(ctr) >= target) return;
  const uint64_t t0 = ptx::globaltimer_ns();
  uint32_t spins = 0;
  while (ld_acquire_u32(ctr) < target) {
    if ((++spins & 0x3ff) == 0 && ptx::globaltimer_ns() - t0 > 4000000000ull) __trap();
  }
}

// fine-grained role stamps of layer 1 (tuning only): slot k of CTA c at trace[ncta * 2 * (nbar + 2) + c * 64 + k], nbar = the
// kernel's grid barriers per step (p.nbar)
// Compiled in only with -DCCB_TUNING (python tools/build.py --tuning): production builds carry no timeline code.
#ifdef CCB_TUNING
#define MEGA_RSTAMP(layer, slot)                                                                         \
  do {                                                                                                   \
    if (p.trace != nullptr && (layer) == 1)                                                              \
      p.trace[static_cast<size_t>(p.ncta) * (2 * (p.nbar + 2)) + static_cast<size_t>(blockIdx.x) * 64 + (slot)] = ptx::globaltimer_ns(); \
  } while (0)
#else
#define MEGA_RSTAMP(layer, slot) do { } while (0)
#endif

// This CTA's share of one GEMM kind (the same in every layer): n units starting at (tile0, kb0), row-tile major.
struct KindSched {
  int n, tile0, kb0, kb;
};

struct ComputeCtx {
  int ct, cw, lane;      // thread / warp index among the compute warps
  int nattn;             // warps per CTA that take attention units
  float* red;            // [2][8] reduction scratch
  int red_it;
  const uint32_t* tbl;   // tile table in shared memory
  const KindSched* sched;
  unsigned* ctr;
  unsigned ncta;
  uint8_t* vs;           // vector-phase scratch (generic pointer) and its shared-window address
  uint32_t vs_u32;
  float* strips;         // [8 warps][192] floats: q (scaled), k_new, v_new of the unit a warp works on
  bool attn_prefetched;  // the first K/V copies of this warp's attention units are already in flight (a_* say which)
  int a_k, a_ib, a_h, a_inflight;  // K/V stream position after the prefetch: unit ordinal, batch, batches issued / in flight
  int u_ctx[4], u_page[4];  // cached tokens / this lane's page id of the warp's first four attention units
  unsigned long long* trace;
  int trace_it;
  unsigned long long* rtrace;   // (tuning) this CTA's 64 role stamps, or null
  int cur_layer;
};

__device__ __forceinline__ float compute_sum(ComputeCtx& cc, float v) {
  v = warp_sum(v);
  float* buf = cc.red + (cc.red_it & 1) * 8;
  cc.red_it++;
  if (cc.lane == 0) buf[cc.cw] = v;
  ptx::named_bar_sync(2, kComputeThreads);
  float r = (cc.lane < 8) ? buf[cc.lane] : 0.f;
  return warp_sum(r);
}

__device__ __forceinline__ void stamp(ComputeCtx& cc) {
#ifdef CCB_TUNING
  if (cc.trace != nullptr && cc.ct == 0) cc.trace[cc.trace_it] = ptx::globaltimer_ns();
  cc.trace_it++;
#else
  (void)cc;
#endif
}

// all compute threads: publish this CTA's global writes of the phase and count the CTA in.  The CTA barrier orders
// every compute thread's stores before thread 0's gpu-scope release (the pattern of a cooperative-groups grid sync).
// The counter is shared by all barriers (barrier #k is complete at (k + 1) * ncta arrivals), so a CTA must never arrive
// at #k+1 before #k is complete: a CTA with GEMM work gets that from its own data dependence (epilogue <- MMA <- X
// tiles <- poll of #k), a CTA without units of a GEMM waits explicitly.
// proxy: this phase's global writes are read through TMA by other CTAs (x / att / mlp rows): fence them into the async proxy
__device__ __forceinline__ void grid_arrive(ComputeCtx& cc, uint32_t xgo_bar, uint32_t helpers_bar = 0, uint32_t helpers_parity = 0,
                                            bool proxy = true) {
  ptx::fence_proxy_async();  // this thread's generic accesses to the X ring (vector scratch) before TMA reuses it
  ptx::named_bar_sync(1, kComputeThreads);
  stamp(cc);
  if (cc.ct == 0) {
    if (helpers_bar != 0) {
      ptx::mbar_wait(helpers_bar, helpers_parity);  // the helper warps' share of the phase is stored
#ifdef CCB_TUNING
      if (cc.rtrace != nullptr && cc.cur_layer == 1) cc.rtrace[44] = ptx::globaltimer_ns();
#endif
    }
    if (proxy) fence_proxy_async_all();  // the global writes are read through TMA (async proxy) by other CTAs
    red_release_add(cc.ctr, 1u);
    if (xgo_bar != 0) ptx::mbar_arrive(xgo_bar);  // the X producer may start polling for this barrier
  }
}
// all compute threads: wait until every CTA has arrived at the first `n` barriers
__device__ __forceinline__ void grid_wait(ComputeCtx& cc, unsigned n) {
  if (cc.ct == 0) poll_counter(cc.ctr, n * cc.ncta);
  ptx::named_bar_sync(1, kComputeThreads);
  stamp(cc);
}

// One warp per (row, head), head_dim 64.  q/k/v = bf16(sum of c_attn partials + bias); the new k/v are appended to
// the cache; softmax(q K^T) V over the cached tokens and the new one.
// The phase is latency bound (8 warps per SM, a few dependent memory round trips each), so the K/V rows travel by
// cp.async into the warp's 8 KB slice of the idle X ring -- no registers are held while they are in flight, which
// keeps ptxas from serialising the loads -- in batches of 16 tokens, two batches in flight; the sum of the c_attn
// partials is computed underneath.  lane = (token group g = lane / 8, 16-byte chunk c = lane % 8); the batches are
// folded with an online softmax.  page_tokens is a power of two (host-checked); offsets are 32-bit element offsets.
// The K/V batches of ALL units of a warp form one stream with two batches in flight: when a unit has no batch left to
// request, the freed half is refilled with the first batches of the warp's next unit, so the fold of q/k/v, the output
// store and the unit change-over run underneath K/V copies (with several units per warp -- 128 / 256 rows -- the phase
// is bound by these copies: 78 MB of K/V per layer at 256 rows).
// prefetch_only: issue the first two batches of the stream and return (called between the arrival at the c_attn
// barrier and the wait for it: cached K/V do not depend on the current step, so their latency hides behind the
// barrier); the phase proper then continues from there (cc.attn_prefetched, cc.a_*).
__device__ __noinline__ void attention_phase(const MegaParams& p, ComputeCtx& cc, int cta, int layer, const float* bias, bool prefetch_only) {
  constexpr int HD = 64;
  const int d = p.d, H = p.H, lane = cc.lane, ncta = p.ncta, cw = cc.cw;
  const int grp = lane >> 3, ch = lane & 7;
  const KvCache cache = p.kv;
  bf16* const att = p.att;
  const int* const ctx_len = p.ctx_len;
  const int* const block_table = p.block_table;
  const float scale = p.scale;
  const uint32_t stage_u32 = cc.vs_u32 + cw * 8192;   // [2 halves][K 16 x 128 B | V 16 x 128 B]
  float* qkvs = cc.strips + cw * 192;
  const int total = p.R * H;
  const int lpt = p.log2_page_tokens, ptm = (1 << lpt) - 1;
  const uint32_t page_stride = static_cast<uint32_t>(H) << (lpt + 6);   // elements per page (all heads)
  const size_t kv_stride = static_cast<size_t>(cache.num_pages) * page_stride;
  const bf16* layer_k = cache.base + static_cast<size_t>(layer) * 2 * kv_stride;
  const uint32_t lane_dst = static_cast<uint32_t>(grp) * 128u + static_cast<uint32_t>(ch) * 16u;
  // Context length and page ids do not change during the step: those of a warp's first four units were loaded once at
  // kernel start (cc.u_ctx / cc.u_page); further units (more than 4 * 11 * ncta units) read theirs when they come up.
  const int maxp = cache.max_pages_per_row;
  const int stride_u = cc.nattn * ncta, unit_first = cw * ncta + cta;
  auto unit_state = [&](int k, int unit, int& ctx, int& page) {
    if (k < 4) {
      ctx = k == 0 ? cc.u_ctx[0] : k == 1 ? cc.u_ctx[1] : k == 2 ? cc.u_ctx[2] : cc.u_ctx[3];
      page = k == 0 ? cc.u_page[0] : k == 1 ? cc.u_page[1] : k == 2 ? cc.u_page[2] : cc.u_page[3];
    } else {
      const int bb = unit / H;
      ctx = ctx_len[bb];
      page = lane < maxp ? block_table[static_cast<uint32_t>(bb) * maxp + lane] : 0;
    }
  };
  // ---- issue side of the K/V stream
  int i_k = 0, i_ib = 0, i_h = 0, inflight = 0;     // unit ordinal, next batch of it, real batches issued / in flight
  int i_ctx = 0, i_page = 0, i_nb = 0;
  bool i_valid = false, i_inwarp = true;
  const bf16* i_kbase = layer_k;
  const int* i_bt = block_table;
  auto issuer_setup = [&](int k) {
    i_k = k;
    i_ib = 0;
    const int unit = unit_first + k * stride_u;
    i_valid = unit < total;
    if (!i_valid) return;
    unit_state(k, unit, i_ctx, i_page);
    const int bb = unit / H, hh = unit - bb * H;
    i_nb = (i_ctx + 15) >> 4;
    i_inwarp = (i_ctx >> lpt) + 1 <= 32;   // page ids held one per lane when they fit a warp, else per-token lookups
    i_kbase = layer_k + (static_cast<uint32_t>(hh) << (lpt + 6)) + ch * 8;  // + page * page_stride + (t & ptm) * 64
    i_bt = block_table + static_cast<uint32_t>(bb) * maxp;
  };
  auto issue_next = [&]() {   // the next batch of the stream into the half it belongs to; always commits a group
    while (i_valid && i_ib >= i_nb) issuer_setup(i_k + 1);
    if (i_valid) {
      const uint32_t dst = stage_u32 + static_cast<uint32_t>(i_h & 1) * 4096u + lane_dst;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int t = i_ib * 16 + i * 4 + grp;
        const bool ok = t < i_ctx;
        const int tt = ok ? t : 0;
        const int page = i_inwarp ? __shfl_sync(0xffffffffu, i_page, tt >> lpt) : i_bt[tt >> lpt];
        const bf16* kp = i_kbase + (static_cast<uint32_t>(page) * page_stride + (static_cast<uint32_t>(tt & ptm) << 6));
        cp_async16(dst + i * 512u, kp, ok ? 16u : 0u);
        cp_async16(dst + i * 512u + 2048u, kp + kv_stride, ok ? 16u : 0u);
      }
      ++i_ib;
      ++i_h;
      ++inflight;
    }
    cp_async_commit();
  };
  if (cc.attn_prefetched) {
    issuer_setup(cc.a_k);
    i_ib = cc.a_ib;
    i_h = cc.a_h;
    inflight = cc.a_inflight;
    cc.attn_prefetched = false;
  } else {
    issuer_setup(0);
    issue_next();
    issue_next();
  }
  if (prefetch_only) {
    cc.attn_prefetched = true;
    cc.a_k = i_k;
    cc.a_ib = i_ib;
    cc.a_h = i_h;
    cc.a_inflight = inflight;
    return;
  }
  int c_h = 0, ui = 0;   // real batches consumed, unit ordinal
#pragma unroll 1
  for (int unit = unit_first; unit < total; unit += stride_u, ++ui) {
    const int b = unit / H, h = unit - b * H;
    int ctx, my_page;
    unit_state(ui, unit, ctx, my_page);
    const int* bt = block_table + static_cast<uint32_t>(b) * maxp;
    const bool pages_in_warp = (ctx >> lpt) + 1 <= 32;
    const bf16* kbase = layer_k + (static_cast<uint32_t>(h) << (lpt + 6)) + ch * 8;
    const int nb = (ctx + 15) >> 4;

    const bool stamp_me = ui == 0 && cw == 1 && lane == 0;   // (tuning) timeline of one unit: slots 32..43 of the role stamps
    if (stamp_me) MEGA_RSTAMP(layer, 32);
    // ---- q / k_new / v_new while the first batches are in flight: lane owns dims (2 lane, 2 lane + 1) of each
    {
      const int rows_out = p.g[0].rows_out, tbl_off = p.g[0].tbl_off;
      const uint32_t* const tbl = cc.tbl;
      const float* const ws = p.ws;
      const uint32_t slot_stride = static_cast<uint32_t>(p.R) * rows_out;
      const int dim = lane * 2;
      const float* src0 = ws + static_cast<uint32_t>(b) * rows_out + h * HD + dim;
      float2 w[3][8];
      int nsl[3];
      // (the bias of this head's q / k / v slices is requested together with the partials: one round trip, not two)
      float2 bqkv[3];
#pragma unroll
      for (int pz = 0; pz < 3; ++pz) bqkv[pz] = __ldg(reinterpret_cast<const float2*>(bias + pz * d + h * HD + dim));
#pragma unroll
      for (int pz = 0; pz < 3; ++pz) {
        nsl[pz] = static_cast<int>(tbl[tbl_off + ((pz * d + h * HD) >> 7)] >> 16);
#pragma unroll
        for (int j = 0; j < 8; ++j)
          w[pz][j] = (j < nsl[pz]) ? ldcg_f2(src0 + pz * d + j * slot_stride) : make_float2(0.f, 0.f);
      }
      float2 part[3];
#pragma unroll
      for (int pz = 0; pz < 3; ++pz) {
        float2 acc = make_float2(0.f, 0.f);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          acc.x += w[pz][j].x; acc.y += w[pz][j].y;
        }
        for (int sl = 8; sl < nsl[pz]; ++sl) {  // (more than 8 contributors per tile: tiny K only)
          const float2 e = ldcg_f2(src0 + pz * d + sl * slot_stride);
          acc.x += e.x; acc.y += e.y;
        }
        const float2 bb = bqkv[pz];
        // the operator-per-kernel path stores c_attn's output as bf16: keep the same rounding
        part[pz] = unpack_bf16x2(pack_bf16x2(acc.x + bb.x, acc.y + bb.y));
      }
      __syncwarp();  // the previous unit's reads of qkvs are complete
      *reinterpret_cast<float2*>(qkvs + dim) = make_float2(part[0].x * scale, part[0].y * scale);
      *reinterpret_cast<float2*>(qkvs + HD + dim) = part[1];
      *reinterpret_cast<float2*>(qkvs + 2 * HD + dim) = part[2];
      __syncwarp();
    }
    if (stamp_me) MEGA_RSTAMP(layer, 33);
    float q8[8], acc[8];
    {
      const float4 a0 = *reinterpret_cast<const float4*>(qkvs + ch * 8), a1 = *reinterpret_cast<const float4*>(qkvs + ch * 8 + 4);
      q8[0] = a0.x; q8[1] = a0.y; q8[2] = a0.z; q8[3] = a0.w; q8[4] = a1.x; q8[5] = a1.y; q8[6] = a1.z; q8[7] = a1.w;
    }
    // the new token: score, and its k / v chunks go to the cache (group 0 writes k, group 1 writes v)
    float m_run, l_run;
    {
      const float4 k0 = *reinterpret_cast<const float4*>(qkvs + HD + ch * 8), k1 = *reinterpret_cast<const float4*>(qkvs + HD + ch * 8 + 4);
      const float4 v0 = *reinterpret_cast<const float4*>(qkvs + 2 * HD + ch * 8), v1 = *reinterpret_cast<const float4*>(qkvs + 2 * HD + ch * 8 + 4);
      float sn = q8[0] * k0.x;
      sn = fmaf(q8[1], k0.y, sn); sn = fmaf(q8[2], k0.z, sn); sn = fmaf(q8[3], k0.w, sn);
      sn = fmaf(q8[4], k1.x, sn); sn = fmaf(q8[5], k1.y, sn); sn = fmaf(q8[6], k1.z, sn); sn = fmaf(q8[7], k1.w, sn);
      sn += __shfl_xor_sync(0xffffffffu, sn, 1);
      sn += __shfl_xor_sync(0xffffffffu, sn, 2);
      sn += __shfl_xor_sync(0xffffffffu, sn, 4);
      m_run = sn;
      const bool g0 = grp == 0;
      l_run = g0 ? 1.f : 0.f;
      acc[0] = g0 ? v0.x : 0.f; acc[1] = g0 ? v0.y : 0.f; acc[2] = g0 ? v0.z : 0.f; acc[3] = g0 ? v0.w : 0.f;
      acc[4] = g0 ? v1.x : 0.f; acc[5] = g0 ? v1.y : 0.f; acc[6] = g0 ? v1.z : 0.f; acc[7] = g0 ? v1.w : 0.f;
      const int page_new = pages_in_warp ? __shfl_sync(0xffffffffu, my_page, ctx >> lpt) : bt[ctx >> lpt];
      if (grp < 2) {
        const float4 s0 = g0 ? k0 : v0, s1 = g0 ? k1 : v1;
        uint4 pk;
        pk.x = pack_bf16x2(s0.x, s0.y); pk.y = pack_bf16x2(s0.z, s0.w); pk.z = pack_bf16x2(s1.x, s1.y); pk.w = pack_bf16x2(s1.z, s1.w);
        const uint32_t off = static_cast<uint32_t>(page_new) * page_stride + (static_cast<uint32_t>(ctx & ptm) << 6);
        *reinterpret_cast<uint4*>(const_cast<bf16*>(kbase) + off + (g0 ? 0 : kv_stride)) = pk;
      }
    }
    if (stamp_me) MEGA_RSTAMP(layer, 34);
    // ---- cached tokens, 16 per batch
#pragma unroll 1
    for (int bi = 0; bi < nb; ++bi) {
      // (groups complete in order: with two batches in flight all but the newest group is enough)
      if (inflight >= 2) cp_async_wait<1>(); else cp_async_wait<0>();
      __syncwarp();
      const uint32_t src = stage_u32 + static_cast<uint32_t>(c_h & 1) * 4096u + lane_dst;
      uint4 kk[4], vv[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        kk[i] = lds_u4(src + i * 512u);
        vv[i] = lds_u4(src + i * 512u + 2048u);
      }
      __syncwarp();                      // every lane has read the half: it may be refilled
      if (stamp_me && bi < 4) MEGA_RSTAMP(layer, 35 + 2 * bi);
      ++c_h;
      --inflight;
      issue_next();
      if (stamp_me && bi < 4) MEGA_RSTAMP(layer, 36 + 2 * bi);                      // this unit's batch bi + 2, or the first batches of the warp's next unit
      float sc[4];
      float m_b = -INFINITY;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float2 k0 = unpack_bf16x2(kk[i].x), k1 = unpack_bf16x2(kk[i].y), k2 = unpack_bf16x2(kk[i].z), k3 = unpack_bf16x2(kk[i].w);
        float s = q8[0] * k0.x;
        s = fmaf(q8[1], k0.y, s); s = fmaf(q8[2], k1.x, s); s = fmaf(q8[3], k1.y, s);
        s = fmaf(q8[4], k2.x, s); s = fmaf(q8[5], k2.y, s); s = fmaf(q8[6], k3.x, s); s = fmaf(q8[7], k3.y, s);
        s += __shfl_xor_sync(0xffffffffu, s, 1);
        s += __shfl_xor_sync(0xffffffffu, s, 2);
        s += __shfl_xor_sync(0xffffffffu, s, 4);
        sc[i] = (bi * 16 + i * 4 + grp < ctx) ? s : -INFINITY;
        m_b = fmaxf(m_b, sc[i]);
      }
      m_b = fmaxf(m_b, __shfl_xor_sync(0xffffffffu, m_b, 8));
      m_b = fmaxf(m_b, __shfl_xor_sync(0xffffffffu, m_b, 16));
      const float m_new = fmaxf(m_run, m_b);
      const float resc = __expf(m_run - m_new);
      m_run = m_new;
      l_run *= resc;
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] *= resc;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float pr = __expf(sc[i] - m_new);  // exp(-inf) = 0 for masked tokens (their V rows were zero-filled)
        l_run += pr;
        const float2 v0 = unpack_bf16x2(vv[i].x), v1 = unpack_bf16x2(vv[i].y), v2 = unpack_bf16x2(vv[i].z), v3 = unpack_bf16x2(vv[i].w);
        acc[0] = fmaf(pr, v0.x, acc[0]); acc[1] = fmaf(pr, v0.y, acc[1]); acc[2] = fmaf(pr, v1.x, acc[2]); acc[3] = fmaf(pr, v1.y, acc[3]);
        acc[4] = fmaf(pr, v2.x, acc[4]); acc[5] = fmaf(pr, v2.y, acc[5]); acc[6] = fmaf(pr, v3.x, acc[6]); acc[7] = fmaf(pr, v3.y, acc[7]);
      }
    }
    if (stamp_me) MEGA_RSTAMP(layer, 43);
    // fold the 4 token groups
    l_run += __shfl_xor_sync(0xffffffffu, l_run, 8);
    l_run += __shfl_xor_sync(0xffffffffu, l_run, 16);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], 8);
      acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], 16);
    }
    if (grp == 0) {
      const float inv = 1.f / l_run;
      uint4 pk;
      pk.x = pack_bf16x2(acc[0] * inv, acc[1] * inv); pk.y = pack_bf16x2(acc[2] * inv, acc[3] * inv);
      pk.z = pack_bf16x2(acc[4] * inv, acc[5] * inv); pk.w = pack_bf16x2(acc[6] * inv, acc[7] * inv);
      *reinterpret_cast<uint4*>(att + static_cast<uint32_t>(b) * d + h * HD + ch * 8) = pk;
    }
  }
}

// attention state of a warp: its unit(s) never change during the step, so context length and page ids are read once
__device__ __forceinline__ void init_attn_ctx(const MegaParams& p, ComputeCtx& cc, int aw, int nattn, int lane, int cta, const uint32_t* tbl,
                                              uint8_t* vs, uint32_t vs_u32, float* strips) {
  cc.cw = aw;
  cc.nattn = nattn;
  cc.lane = lane;
  cc.tbl = tbl;
  cc.vs = vs;
  cc.vs_u32 = vs_u32;
  cc.strips = strips;
  cc.attn_prefetched = false;
  cc.a_k = cc.a_ib = cc.a_h = cc.a_inflight = 0;
  cc.rtrace = p.trace ? p.trace + static_cast<size_t>(p.ncta) * (2 * (p.nbar + 2)) + static_cast<size_t>(cta) * 64 : nullptr;
  cc.cur_layer = 0;
#pragma unroll
  for (int ui = 0; ui < 4; ++ui) {
    const int unit = (aw + nattn * ui) * p.ncta + cta;
    cc.u_ctx[ui] = 0;
    cc.u_page[ui] = 0;
    if (unit < p.R * p.H) {
      const int b = unit / p.H;
      cc.u_ctx[ui] = p.ctx_len[b];
      cc.u_page[ui] = lane < p.kv.max_pages_per_row ? p.block_table[static_cast<uint32_t>(b) * p.kv.max_pages_per_row + lane] : 0;
    }
  }
}

// The X-producer, MMA and TMEM-allocator warps have nothing to do while the attention phase runs: each takes the
// attention units of one more "compute warp" (11 instead of 8 warps: GPT2-XL x 64 rows = 1600 units on 148 x 11 warps,
// one unit per warp instead of two for a third of them).  Their K/V staging lies behind the X ring (up to ~170 rows), so
// they prefetch as soon as they get here; vgo = c_attn complete everywhere, vdone = this warp's outputs are stored.
__device__ __forceinline__ void helper_attention(const MegaParams& p, ComputeCtx& hc, int cta, int l, uint32_t vgo, uint32_t vdone,
                                                 bool early_prefetch) {
  const float* bias = p.layers[l].b_qkv;
  // The helpers get here while this CTA's c_attn MMAs may still be reading the X ring.  Their K/V staging (slices 8..10
  // of the vector scratch, 64..88 KB from the ring's start) lies behind the ring only while the ring is <= 64 KB; above
  // ~170 rows (three tiles of > 21 KB) it is inside it, and an early prefetch would overwrite live activation tiles
  // (seen as run-to-run differences of sampled / beam captions at >= 200 rows): then the copies start after vgo.
  if (early_prefetch) attention_phase(p, hc, cta, l, bias, true);
  ptx::mbar_wait(vgo, static_cast<uint32_t>(l) & 1u);
  if (hc.lane == 0 && hc.cw == 8) MEGA_RSTAMP(l, 48);
  attention_phase(p, hc, cta, l, bias, false);
  fence_proxy_async_all();   // att rows are fetched by other CTAs through TMA
  __syncwarp();
  if (hc.lane == 0) {
    MEGA_RSTAMP(l, 45 + hc.cw - 8);
    ptx::mbar_arrive(vdone);
  }
}

// h[t] = (embed | h[t] + bias + sum of split-K partials); x[t] = LayerNorm(h[t]) for the rows t = cta, cta + ncta, ...
// The row is staged in shared memory (each thread re-reads only what it wrote).
__device__ __noinline__ void ln_phase(const MegaParams& p, ComputeCtx& cc, int cta, bool embed, int prev_kind, const float* prev_bias,
                                      const float* gamma, const float* beta) {
  const int d = p.d, nq = d >> 2, R = p.R, ncta = p.ncta;
  float4* rowbuf = reinterpret_cast<float4*>(cc.vs);
  const uint32_t* const tbl = cc.tbl;
  const float* const ws = p.ws;
  float* const hbase = p.h;
  bf16* const xbase = p.x;
  const float eps = p.eps;
  const int ct = cc.ct;
  const int p_tbl_off = p.g[prev_kind].tbl_off, p_rows_out = p.g[prev_kind].rows_out;
  for (int t = cta; t < R; t += ncta) {
    float s = 0.f;
    float4* hrow = reinterpret_cast<float4*>(hbase + static_cast<size_t>(t) * d);
    if (embed) {
      const int tok = p.tokens[t];
      const uint2* te = reinterpret_cast<const uint2*>(p.wte + static_cast<size_t>(tok) * d);
      const uint2* pe = p.wpe ? reinterpret_cast<const uint2*>(p.wpe + static_cast<size_t>(p.ctx_len[t]) * d) : nullptr;
#pragma unroll 1
      for (int q = ct; q < nq; q += kComputeThreads) {
        const uint2 e = __ldg(te + q);
        const float2 e0 = unpack_bf16x2(e.x), e1 = unpack_bf16x2(e.y);
        float4 a = make_float4(e0.x, e0.y, e1.x, e1.y);
        if (pe != nullptr) {
          const uint2 w = __ldg(pe + q);
          const float2 w0 = unpack_bf16x2(w.x), w1 = unpack_bf16x2(w.y);
          a.x += w0.x; a.y += w0.y; a.z += w1.x; a.w += w1.y;
        }
        hrow[q] = a;
        rowbuf[q] = a;
        s += (a.x + a.y) + (a.z + a.w);
      }
    } else {
      // two columns (float4) per thread per pass, their slot loads issued together: the phase is a chain of L2
      // round trips, so the fewer dependent ones the better
      const uint32_t slot_stride = static_cast<uint32_t>(R) * p_rows_out;
      const float* src = ws + static_cast<uint32_t>(t) * p_rows_out;
#pragma unroll 1
      for (int q0 = ct; q0 < nq; q0 += 2 * kComputeThreads) {
        const int q1 = q0 + kComputeThreads;
        const bool has1 = q1 < nq;
        const int nsl0 = static_cast<int>(tbl[p_tbl_off + (q0 >> 5)] >> 16);
        const int nsl1 = has1 ? static_cast<int>(tbl[p_tbl_off + (q1 >> 5)] >> 16) : 0;
        const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
        const float4 b0 = __ldg(reinterpret_cast<const float4*>(prev_bias) + q0);
        const float4 b1 = has1 ? __ldg(reinterpret_cast<const float4*>(prev_bias) + q1) : z4;
        const float4 r0 = hrow[q0];
        const float4 r1 = has1 ? hrow[q1] : z4;
        float4 a0 = z4, a1 = z4;
        const int nmax = nsl0 > nsl1 ? nsl0 : nsl1;
#pragma unroll 1
        for (int s0 = 0; s0 < nmax; s0 += kLnSlots) {
          // all slots of both columns in flight at once (c_proj / mlp.c_proj tiles have ~13 contributors on 148 SMs)
          float4 w0[kLnSlots], w1[kLnSlots];
#pragma unroll
          for (int j = 0; j < kLnSlots; ++j) w0[j] = (s0 + j < nsl0) ? ldcg_f4(src + (q0 << 2) + (s0 + j) * slot_stride) : z4;
#pragma unroll
          for (int j = 0; j < kLnSlots; ++j) w1[j] = (s0 + j < nsl1) ? ldcg_f4(src + (q1 << 2) + (s0 + j) * slot_stride) : z4;
#pragma unroll
          for (int j = 0; j < kLnSlots; ++j) {
            a0.x += w0[j].x; a0.y += w0[j].y; a0.z += w0[j].z; a0.w += w0[j].w;
          }
#pragma unroll
          for (int j = 0; j < kLnSlots; ++j) {
            a1.x += w1[j].x; a1.y += w1[j].y; a1.z += w1[j].z; a1.w += w1[j].w;
          }
        }
        const float4 o0 = make_float4(r0.x + (a0.x + b0.x), r0.y + (a0.y + b0.y), r0.z + (a0.z + b0.z), r0.w + (a0.w + b0.w));
        hrow[q0] = o0;
        rowbuf[q0] = o0;
        s += (o0.x + o0.y) + (o0.z + o0.w);
        if (has1) {
          const float4 o1 = make_float4(r1.x + (a1.x + b1.x), r1.y + (a1.y + b1.y), r1.z + (a1.z + b1.z), r1.w + (a1.w + b1.w));
          hrow[q1] = o1;
          rowbuf[q1] = o1;
          s += (o1.x + o1.y) + (o1.z + o1.w);
        }
      }
    }
    const float mean = compute_sum(cc, s) / d;
    float qv = 0.f;
#pragma unroll 1
    for (int q = ct; q < nq; q += kComputeThreads) {
      const float4 v = rowbuf[q];
      const float a = v.x - mean, b = v.y - mean, c2 = v.z - mean, d2 = v.w - mean;
      qv += (a * a + b * b) + (c2 * c2 + d2 * d2);
    }
    // gamma / beta of (up to) two columns are requested before the second reduction
    const int qa = ct, qb = ct + kComputeThreads;
    const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
    const float4 ga = qa < nq ? __ldg(reinterpret_cast<const float4*>(gamma) + qa) : z4;
    const float4 ba = qa < nq ? __ldg(reinterpret_cast<const float4*>(beta) + qa) : z4;
    const float4 gb = qb < nq ? __ldg(reinterpret_cast<const float4*>(gamma) + qb) : z4;
    const float4 bb = qb < nq ? __ldg(reinterpret_cast<const float4*>(beta) + qb) : z4;
    const float var = compute_sum(cc, qv) / d;
    const float rstd = rsqrtf(var + eps);
    uint2* xr = reinterpret_cast<uint2*>(xbase + static_cast<size_t>(t) * d);
#pragma unroll 1
    for (int q = ct; q < nq; q += kComputeThreads) {
      const float4 v = rowbuf[q];
      const float4 g4 = q == qa ? ga : q == qb ? gb : __ldg(reinterpret_cast<const float4*>(gamma) + q);
      const float4 b4 = q == qa ? ba : q == qb ? bb : __ldg(reinterpret_cast<const float4*>(beta) + q);
      uint2 pk;
      pk.x = pack_bf16x2((v.x - mean) * rstd * g4.x + b4.x, (v.y - mean) * rstd * g4.y + b4.y);
      pk.y = pack_bf16x2((v.z - mean) * rstd * g4.z + b4.z, (v.w - mean) * rstd * g4.w + b4.w);
      xr[q] = pk;
    }
  }
}

// mlp[t, f] = gelu_new(sum of c_fc partials + bias)
// A thread owns up to three float4 items (64 rows x 6400 features on 148 x 256 threads = 2.7 per thread).  The phase is
// a chain of L2 round trips, so the slot loads of ALL its items are issued before the first one is used (one round trip
// instead of one per item).
__device__ __noinline__ void gelu_phase(const MegaParams& p, ComputeCtx& cc, int cta, const float* bias) {
  constexpr int kItems = 3, kSl = 4;
  const uint32_t rows_out = p.g[2].rows_out, tbl_off = p.g[2].tbl_off;
  const uint32_t nq = rows_out >> 2;
  const uint32_t total = static_cast<uint32_t>(p.R) * nq;
  const uint32_t slot_stride = static_cast<uint32_t>(p.R) * rows_out;
  const uint32_t step = static_cast<uint32_t>(p.ncta) * kComputeThreads;
  const uint32_t* const tbl = cc.tbl;
  const float* const ws = p.ws;
  bf16* const mlp = p.mlp;
  const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 1
  for (uint32_t idx0 = static_cast<uint32_t>(cta) * kComputeThreads + cc.ct; idx0 < total; idx0 += kItems * step) {
    float4 w[kItems][kSl], b[kItems];
    uint32_t off[kItems], q[kItems];
    int nsl[kItems];
#pragma unroll
    for (int j = 0; j < kItems; ++j) {
      const uint32_t idx = idx0 + j * step;
      const bool ok = idx < total;
      const uint32_t t = ok ? idx / nq : 0u;
      q[j] = ok ? idx - t * nq : 0u;
      off[j] = t * rows_out + (q[j] << 2);
      nsl[j] = ok ? static_cast<int>(tbl[tbl_off + (q[j] >> 5)] >> 16) : -1;
#pragma unroll
      for (int sl = 0; sl < kSl; ++sl) w[j][sl] = (sl < nsl[j]) ? ldcg_f4(ws + off[j] + sl * slot_stride) : z4;
      b[j] = __ldg(reinterpret_cast<const float4*>(bias) + q[j]);
    }
#pragma unroll
    for (int j = 0; j < kItems; ++j) {
      if (nsl[j] < 0) continue;
      float4 acc = z4;
#pragma unroll
      for (int sl = 0; sl < kSl; ++sl) {   // slot order (absent slots add zero)
        acc.x += w[j][sl].x; acc.y += w[j][sl].y; acc.z += w[j][sl].z; acc.w += w[j][sl].w;
      }
      for (int sl = kSl; sl < nsl[j]; ++sl) {  // (more than four contributors per tile: small K only)
        const float4 e = ldcg_f4(ws + off[j] + sl * slot_stride);
        acc.x += e.x; acc.y += e.y; acc.z += e.z; acc.w += e.w;
      }
      float o[4] = {acc.x + b[j].x, acc.y + b[j].y, acc.z + b[j].z, acc.w + b[j].w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        // same form as the GEMM epilogue's gelu_new: 0.5 x (1 + tanh(u)) == x - x / (1 + exp(2u))
        const float xx = o[k];
        const float u = 0.7978845608028654f * (xx + 0.044715f * xx * xx * xx);
        o[k] = xx - __fdividef(xx, 1.f + __expf(2.f * u));
      }
      uint2 pk;
      pk.x = pack_bf16x2(o[0], o[1]);
      pk.y = pack_bf16x2(o[2], o[3]);
      *reinterpret_cast<uint2*>(mlp + off[j]) = pk;
    }
  }
}


// LayerNorm gains / offsets and the four bias vectors of a layer are read once per step and would come from HBM in the
// middle of a latency-bound phase (a DRAM round trip is ~1 us here): the otherwise idle TMEM-owner warps of all CTAs
// pull them into L2 one layer ahead, 128 bytes per lane.
__device__ __forceinline__ void prefetch_layer_vectors(const MegaParams& p, int l, int cta, int lane) {
  const MegaLayer ly = p.layers[l];
  const float* vec[8] = {ly.ln1_g, ly.ln1_b, ly.b_qkv, ly.b_proj, ly.ln2_g, ly.ln2_b, ly.b_fc, ly.b_fc2};
  const int len[8] = {p.d, p.d, 3 * p.d, p.d, p.d, p.d, p.ff, p.d};
  const int step = p.ncta * 32;
#pragma unroll
  for (int v = 0; v < 8; ++v)
    for (int i = (cta * 32 + lane) * 32; i < len[v]; i += step * 32)
      asm volatile("prefetch.global.L2 [%0];" ::"l"(vec[v] + i));
}

struct EpiCtx {
  uint32_t tmem_base, t_full0, t_empty0;  // barrier b at +8 b
  uint32_t ait;                           // accumulator buffers consumed so far
};

// TMEM accumulator -> fp32 split-K partial in the workspace, for every segment of this CTA in GEMM `kind`.
// Compute warp w reads TMEM lane quadrant w % 4 (its hardware-accessible quarter) and column half w / 4.
__device__ __noinline__ void epilogue_phase(const MegaParams& p, ComputeCtx& cc, EpiCtx& ec, int cta, int kind, int layer) {
  // every field used below is copied to a register first: the partial stores could alias anything reached through
  // the references, and a reload per store costs more than the store
  const int rows_out = p.g[kind].rows_out, tbl_off = p.g[kind].tbl_off;
  const int R = p.R, N = p.N;
  float* const ws = p.ws;
  const uint32_t* const tbl = cc.tbl;
  const KindSched sc = cc.sched[kind];
  const uint32_t tmem_base = ec.tmem_base, t_full0 = ec.t_full0, t_empty0 = ec.t_empty0;
  uint32_t ait = ec.ait;
  const int lane = cc.lane, quad = cc.cw & 3, half = cc.cw >> 2;
  const bool stamp0 = cc.ct == 0;
  const int c_beg = half * (N >> 1);
  int c_end = (half + 1) * (N >> 1);
  if (c_end > R) c_end = R;
  const bool wide = ((N >> 1) & 31) == 0;
  int n = sc.n, tile = sc.tile0, kb = sc.kb0;
#pragma unroll 1
  while (n > 0) {
    int len = sc.kb - kb;
    if (len > n) len = n;
    const uint32_t buf = ait & 1, aph = (ait >> 1) & 1;
    ++ait;
    ptx::mbar_wait(t_full0 + 8u * buf, aph);
    ptx::tc_fence_after();
    if (stamp0) MEGA_RSTAMP(layer, kind * 8 + 4);
    const int slot = cta - static_cast<int>(tbl[tbl_off + tile] & 0xffffu);
    const int i = tile * 128 + quad * 32 + lane;
    const bool i_ok = i < rows_out;
    float* dst = ws + (static_cast<size_t>(slot) * R + c_beg) * rows_out + i;
    const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + buf * static_cast<uint32_t>(N);
    if (wide) {
#pragma unroll 1
      for (int c0 = c_beg; c0 < c_end; c0 += 32) {
        uint32_t r[32];
        ptx::tmem_ld32(taddr + c0, r);
        ptx::tmem_ld_wait();
        if (i_ok) {
          if (c0 + 32 <= c_end) {
#pragma unroll
            for (int v = 0; v < 32; ++v) dst[static_cast<size_t>(v) * rows_out] = __uint_as_float(r[v]);
          } else {
#pragma unroll
            for (int v = 0; v < 32; ++v)
              if (c0 + v < c_end) dst[static_cast<size_t>(v) * rows_out] = __uint_as_float(r[v]);
          }
        }
        dst += static_cast<size_t>(32) * rows_out;
      }
    } else {
#pragma unroll 1
      for (int c0 = c_beg; c0 < c_end; c0 += 8) {
        uint32_t r[8];
        ptx::tmem_ld8(taddr + c0, r);
        ptx::tmem_ld_wait();
        if (i_ok) {
#pragma unroll
          for (int v = 0; v < 8; ++v)
            if (c0 + v < c_end) dst[static_cast<size_t>(v) * rows_out] = __uint_as_float(r[v]);
        }
        dst += static_cast<size_t>(8) * rows_out;
      }
    }
    ptx::tc_fence_before();
    __syncwarp();
    if (lane == 0) ptx::mbar_arrive(t_empty0 + 8u * buf);
    if (stamp0) MEGA_RSTAMP(layer, kind * 8 + 5);
    n -= len;
    kb = 0;
    ++tile;
  }
  ec.ait = ait;
}

__global__ void __launch_bounds__(kThreads, 1) decode_mega_kernel(const __grid_constant__ CUtensorMap xmap_x,
                                                                  const __grid_constant__ CUtensorMap xmap_att,
                                                                  const __grid_constant__ CUtensorMap xmap_mlp,
                                                                  const __grid_constant__ MegaParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_u32 = ptx::smem_u32(smem_raw);
  const uint32_t base = (raw_u32 + 1023u) & ~1023u;
  uint8_t* gen = smem_raw + (base - raw_u32);
  const int nW = p.nW, nX = p.nX;
  const int grp = p.grp;   // units per ring hand-over: 2 (slot pairs) or 1 (256 rows: the X ring holds only three tiles)
  const uint32_t xstage = static_cast<uint32_t>(p.N) * 128u;
  const uint32_t w_ring = base;
  const uint32_t x_ring = w_ring + nW * kWStage;
  // after the X ring / vector scratch (>= kVecScratch bytes): q/k/v strips (11 x 192 floats), reduction scratch,
  // schedule, tile table, barriers
  const uint32_t misc_off = nW * kWStage + p.xring_bytes;
  float* strips = reinterpret_cast<float*>(gen + misc_off);
  float* red = reinterpret_cast<float*>(gen + misc_off + kAttnWarps * 192 * 4);
  KindSched* sched = reinterpret_cast<KindSched*>(gen + misc_off + kAttnWarps * 192 * 4 + 64);
  uint32_t* tbl = reinterpret_cast<uint32_t*>(gen + misc_off + kAttnWarps * 192 * 4 + 64 + 64);
  const uint32_t bar_off = misc_off + kAttnWarps * 192 * 4 + 64 + 64 + kTblMax * 4;
  const uint32_t bars = base + bar_off;
  // barrier layout: w_full[nW], w_empty[nW], x_full[nX], x_empty[nX], t_full[2], t_empty[2], xgo, tmem slot
  const uint32_t w_full0 = bars, w_empty0 = bars + 8u * nW;
  const uint32_t x_full0 = bars + 16u * nW, x_empty0 = x_full0 + 8u * nX;
  const uint32_t t_full0 = x_empty0 + 8u * nX, t_empty0 = t_full0 + 16u;
  const uint32_t xgo = t_empty0 + 16u;  // compute -> X producer: "this CTA arrived at the barrier you need"
  const uint32_t vgo = xgo + 8u;        // compute -> helper warps: "c_attn is complete everywhere: attention may start"
  const uint32_t vdone = vgo + 8u;      // helper warps -> compute: "my attention unit of this layer is stored"
  const uint32_t tmem_slot = vdone + 8u;
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(gen + (tmem_slot - base));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int cta = blockIdx.x, ncta = p.ncta;

  if (threadIdx.x == 0) {
    for (int s = 0; s < nW; ++s) {
      ptx::mbar_init(w_full0 + 8u * s, 1);
      ptx::mbar_init(w_empty0 + 8u * s, 1);
    }
    for (int s = 0; s < nX; ++s) {
      ptx::mbar_init(x_full0 + 8u * s, 1);
      ptx::mbar_init(x_empty0 + 8u * s, 1);
    }
    for (int b = 0; b < 2; ++b) {
      ptx::mbar_init(t_full0 + 8u * b, 1);
      ptx::mbar_init(t_empty0 + 8u * b, 8);
    }
    ptx::mbar_init(xgo, 1);
    ptx::mbar_init(vgo, 1);
    ptx::mbar_init(vdone, 3);
    ptx::fence_mbar_init();
  }
  if (threadIdx.x >= 32 && threadIdx.x < 36) {
    const int kind = threadIdx.x - 32;
    const MegaGemmShape& g = p.g[kind];
    // few units (small models): only the first `units` CTAs take part, so that the contributors of a row tile
    // are consecutive CTAs (slot = cta - first contributor)
    const int nc = g.units < ncta ? g.units : ncta;
    const int u0 = cta < nc ? static_cast<int>(static_cast<long long>(cta) * g.units / nc) : 0;
    const int u1 = cta < nc ? static_cast<int>(static_cast<long long>(cta + 1) * g.units / nc) : 0;
    KindSched k;
    k.n = u1 - u0;
    k.tile0 = u0 / g.kb;
    k.kb0 = u0 - k.tile0 * g.kb;
    k.kb = g.kb;
    sched[kind] = k;
  }
  if (warp == 3) ptx::tmem_alloc<512>(tmem_slot);
  for (int i = threadIdx.x; i < p.tbl_entries; i += kThreads) tbl[i] = p.tile_tbl[i];
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;
  const bool helper_prefetch = static_cast<uint32_t>(nX) * xstage <= 8u * 8192u;   // (see helper_attention)

  if (warp == 0) {
    // ------------------------------------------------------------------ W producer
    // (the whole warp walks the schedule and waits; one elected lane issues: converged code lets the compiler emit
    //  the single-thread instructions without a per-instruction election loop)
    // Ring slots are handed over in PAIRS (two consecutive units of this CTA's stream share one full / empty barrier):
    // half the waits, expect_tx and commits per byte in all three role loops, which are what paces a GEMM phase.
    uint32_t sp = 0, ph = 0;   // slot pair, its phase
    const uint32_t nWp = static_cast<uint32_t>(nW / grp);
#pragma unroll 1
    for (int l = 0; l < p.L; ++l) {
#pragma unroll 1
      for (int kind = 0; kind < 4; ++kind) {
        const CUtensorMap* wm = p.wmaps + (l * 4 + kind);
        const KindSched sc = sched[kind];
        int tile = sc.tile0, kb = sc.kb0;
#pragma unroll 1
        for (int n = sc.n; n > 0; n -= grp) {
          const bool two = grp == 2 && n > 1;
          ptx::mbar_wait(w_empty0 + 8u * sp, ph ^ 1);
          if (ptx::elect_one()) {
            const uint32_t full = w_full0 + 8u * sp;
            ptx::mbar_arrive_expect_tx(full, two ? 2 * kWStage : kWStage);
            ptx::tma_load_2d(w_ring + (grp * sp) * kWStage, wm, full, kb * 64, tile * 128, ptx::kEvictFirst);
            int kb2 = kb + 1, tile2 = tile;
            if (kb2 == sc.kb) { kb2 = 0; ++tile2; }
            if (two) ptx::tma_load_2d(w_ring + (grp * sp + 1) * kWStage, wm, full, kb2 * 64, tile2 * 128, ptx::kEvictFirst);
          }
          __syncwarp();
          if (++sp == nWp) { sp = 0; ph ^= 1; }
          kb += grp;
          while (kb >= sc.kb) { kb -= sc.kb; ++tile; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ X producer (+ attention helper)
    ComputeCtx hc;
    init_attn_ctx(p, hc, 8, kAttnWarps, lane, cta, tbl, gen + nW * kWStage, x_ring, strips);
    uint32_t s = 0, ph = 0;
#pragma unroll 1
    for (int l = 0; l < p.L; ++l) {
#pragma unroll 1
      for (int kind = 0; kind < 4; ++kind) {
        if (kind == 1) helper_attention(p, hc, cta, l, vgo, vdone, helper_prefetch);   // between the c_attn and the c_proj tiles
        const CUtensorMap* xm = (kind == 1) ? &xmap_att : (kind == 3) ? &xmap_mlp : &xmap_x;
        const KindSched sc = sched[kind];
        if (sc.n == 0) continue;
        // the activation is complete once every CTA passed barrier #(8l + 2 kind) (the vector phase before it);
        // no point in polling before this CTA's own compute warps arrived there (their (4l + kind)-th signal)
        ptx::mbar_wait(xgo, static_cast<uint32_t>(4 * l + kind) & 1u);
        if (lane == 0) {
          poll_counter(p.sync, static_cast<unsigned>(8 * l + 2 * kind + 1) * ncta);
          fence_proxy_async_all();
          MEGA_RSTAMP(l, kind * 8 + 0);
        }
        __syncwarp();
        int kb = sc.kb0;
#pragma unroll 1
        for (int n = sc.n; n > 0; n -= grp) {
          const bool two = grp == 2 && n > 1;
          ptx::mbar_wait(x_empty0 + 8u * s, ph ^ 1);
          if (lane == 0) {
            const uint32_t full = x_full0 + 8u * s;
            ptx::mbar_arrive_expect_tx(full, two ? 2 * xstage : xstage);
            ptx::tma_load_2d(x_ring + (grp * s) * xstage, xm, full, kb * 64, 0, ptx::kEvictLast);
            int kb2 = kb + 1;
            if (kb2 == sc.kb) kb2 = 0;
            if (two) ptx::tma_load_2d(x_ring + (grp * s + 1) * xstage, xm, full, kb2 * 64, 0, ptx::kEvictLast);
          }
          __syncwarp();
          if (++s == static_cast<uint32_t>(nX / grp)) { s = 0; ph ^= 1; }
          kb += grp;
          while (kb >= sc.kb) kb -= sc.kb;
        }
        if (lane == 0) MEGA_RSTAMP(l, kind * 8 + 1);
      }
    }
  } else if (warp == 2) {
    // ------------------------------------------------------------------ MMA issuer (+ attention helper)
    ComputeCtx hc;
    init_attn_ctx(p, hc, 9, kAttnWarps, lane, cta, tbl, gen + nW * kWStage, x_ring, strips);
    // The issue loop is instruction bound (one warp, dependent address arithmetic in front of every tcgen05.mma), so
    // it works on slot PAIRS: one set of waits, one descriptor computation (kept incrementally, no multiplies) and
    // one pair of ring commits per two units; the segment bookkeeping of both units is done ahead of the waits.
    const uint32_t idesc = ptx::umma_idesc_bf16(128, p.N);
    const uint64_t wdesc0 = ptx::umma_desc_k_sw128(w_ring), xdesc0 = ptx::umma_desc_k_sw128(x_ring);
    const uint64_t wstep = static_cast<uint64_t>(kWStage >> 4), xstep = static_cast<uint64_t>(xstage >> 4);
    uint64_t wd = wdesc0, xd = xdesc0;                    // descriptors of the current slot pair
    uint32_t ws = 0, wph = 0, xs = 0, xph = 0, ait = 0;   // slot PAIRS and their phases
    const uint32_t nWp = static_cast<uint32_t>(nW / grp), nXp = static_cast<uint32_t>(nX / grp);
    const uint32_t nacc = static_cast<uint32_t>(p.N);
#pragma unroll 1
    for (int l = 0; l < p.L; ++l) {
#pragma unroll 1
      for (int kind = 0; kind < 4; ++kind) {
        if (kind == 1) helper_attention(p, hc, cta, l, vgo, vdone, helper_prefetch);   // all c_attn MMAs of this CTA are issued
        const KindSched sc = sched[kind];
        int kb = sc.kb0;          // k block of the next unit inside its row tile
        int seg_left = 0;         // units left in the current segment (0: the next unit opens one)
        uint32_t buf = 0;
#pragma unroll 1
        for (int n = sc.n; n > 0; n -= grp) {
          const bool two = grp == 2 && n > 1;
          // ---- segment bookkeeping of both units (a segment = the rest of a row tile or of this CTA's range)
          bool first0 = false, first1 = false;
          if (seg_left == 0) {
            seg_left = sc.kb - kb;
            if (seg_left > n) seg_left = n;
            buf = ait & 1;
            ptx::mbar_wait(t_empty0 + 8u * buf, ((ait >> 1) & 1) ^ 1);
            ++ait;
            first0 = true;
          }
          const uint32_t buf0 = buf;
          const bool end0 = --seg_left == 0;
          if (++kb == sc.kb) kb = 0;
          bool end1 = false;
          if (two) {
            if (seg_left == 0) {
              seg_left = sc.kb - kb;
              if (seg_left > n - 1) seg_left = n - 1;
              buf = ait & 1;
              ptx::mbar_wait(t_empty0 + 8u * buf, ((ait >> 1) & 1) ^ 1);
              ++ait;
              first1 = true;
            }
            end1 = --seg_left == 0;
            if (++kb == sc.kb) kb = 0;
          }
          const uint32_t buf1 = buf;
          ptx::mbar_wait(w_full0 + 8u * ws, wph);
          ptx::mbar_wait(x_full0 + 8u * xs, xph);
          ptx::tc_fence_after();
          if (ptx::elect_one()) {
            if (first0) MEGA_RSTAMP(l, kind * 8 + 2);
            const uint32_t tacc0 = tmem_base + buf0 * nacc;
            ptx::umma_bf16(tacc0, wd, xd, idesc, first0 ? 0u : 1u);
            ptx::umma_bf16(tacc0, wd + 2u, xd + 2u, idesc, 1u);
            ptx::umma_bf16(tacc0, wd + 4u, xd + 4u, idesc, 1u);
            ptx::umma_bf16(tacc0, wd + 6u, xd + 6u, idesc, 1u);
            if (end0) ptx::umma_commit(t_full0 + 8u * buf0);
            if (two) {
              const uint32_t tacc1 = tmem_base + buf1 * nacc;
              const uint64_t wd1 = wd + wstep, xd1 = xd + xstep;
              ptx::umma_bf16(tacc1, wd1, xd1, idesc, first1 ? 0u : 1u);
              ptx::umma_bf16(tacc1, wd1 + 2u, xd1 + 2u, idesc, 1u);
              ptx::umma_bf16(tacc1, wd1 + 4u, xd1 + 4u, idesc, 1u);
              ptx::umma_bf16(tacc1, wd1 + 6u, xd1 + 6u, idesc, 1u);
              if (end1) ptx::umma_commit(t_full0 + 8u * buf1);
            }
            ptx::umma_commit(w_empty0 + 8u * ws);
            ptx::umma_commit(x_empty0 + 8u * xs);
            if (n <= grp) MEGA_RSTAMP(l, kind * 8 + 3);
          }
          __syncwarp();
          wd += grp * wstep;
          xd += grp * xstep;
          if (++ws == nWp) { ws = 0; wph ^= 1; wd = wdesc0; }
          if (++xs == nXp) { xs = 0; xph ^= 1; xd = xdesc0; }
        }
      }
    }
  } else if (warp == 3) {
    // ------------------------------------------------------------------ TMEM owner: attention helper only
    ComputeCtx hc;
    init_attn_ctx(p, hc, 10, kAttnWarps, lane, cta, tbl, gen + nW * kWStage, x_ring, strips);
    prefetch_layer_vectors(p, 0, cta, lane);
    for (int l = 0; l < p.L; ++l) {
      if (l + 1 < p.L) prefetch_layer_vectors(p, l + 1, cta, lane);
      helper_attention(p, hc, cta, l, vgo, vdone, helper_prefetch);
    }
  } else if (warp >= kComputeWarp0) {
    // ------------------------------------------------------------------ compute warps
    ComputeCtx cc;
    cc.ct = threadIdx.x - kComputeWarp0 * 32;
    cc.cw = warp - kComputeWarp0;
    cc.lane = lane;
    cc.red = red;
    cc.red_it = 0;
    cc.tbl = tbl;
    cc.sched = sched;
    cc.ctr = p.sync;
    cc.ncta = ncta;
    cc.vs = gen + nW * kWStage;
    cc.vs_u32 = x_ring;
    cc.strips = strips;
    cc.trace = p.trace ? p.trace + static_cast<size_t>(cta) * (2 * (p.nbar + 2)) : nullptr;
    cc.trace_it = 0;
    init_attn_ctx(p, cc, warp - kComputeWarp0, kAttnWarps, lane, cta, tbl, gen + nW * kWStage, x_ring, strips);
    EpiCtx ec;
    ec.tmem_base = tmem_base;
    ec.t_full0 = t_full0;
    ec.t_empty0 = t_empty0;
    ec.ait = 0;

#pragma unroll 1
    for (int l = 0; l < p.L; ++l) {
      const MegaLayer ly = p.layers[l];
      cc.cur_layer = l;
      if (l > 0) grid_wait(cc, 8 * l);
      ln_phase(p, cc, cta, l == 0, 3, l > 0 ? p.layers[l - 1].b_fc2 : nullptr, ly.ln1_g, ly.ln1_b);
      grid_arrive(cc, xgo);     // #8l
      epilogue_phase(p, cc, ec, cta, 0, l);
      if (sched[0].n == 0) grid_wait(cc, 8 * l + 1);  // (see grid_arrive: no arrival at #k+1 before #k is complete)
      grid_arrive(cc, 0, 0, 0, false);       // #8l+1 (split-K partials: read with ld.global.cg, no TMA consumer)
      // (warp 0 polls the barrier for the CTA: it goes straight to the wait and fetches its K/V afterwards)
      if (cc.cw != 0) attention_phase(p, cc, cta, l, ly.b_qkv, true);
      grid_wait(cc, 8 * l + 2);
      if (cc.ct == 0) ptx::mbar_arrive(vgo);   // the helper warps start their units
      attention_phase(p, cc, cta, l, ly.b_qkv, false);
      if (lane == 0) MEGA_RSTAMP(l, 50 + cc.cw);
      grid_arrive(cc, xgo, vdone, static_cast<uint32_t>(l) & 1u);     // #8l+2
      epilogue_phase(p, cc, ec, cta, 1, l);
      if (sched[1].n == 0) grid_wait(cc, 8 * l + 3);  // (see grid_arrive: no arrival at #k+1 before #k is complete)
      grid_arrive(cc, 0, 0, 0, false);       // #8l+3 (split-K partials: read with ld.global.cg, no TMA consumer)
      grid_wait(cc, 8 * l + 4);
      ln_phase(p, cc, cta, false, 1, ly.b_proj, ly.ln2_g, ly.ln2_b);
      grid_arrive(cc, xgo);     // #8l+4
      epilogue_phase(p, cc, ec, cta, 2, l);
      if (sched[2].n == 0) grid_wait(cc, 8 * l + 5);  // (see grid_arrive: no arrival at #k+1 before #k is complete)
      grid_arrive(cc, 0, 0, 0, false);       // #8l+5 (split-K partials: read with ld.global.cg, no TMA consumer)
      grid_wait(cc, 8 * l + 6);
      gelu_phase(p, cc, cta, ly.b_fc);
      grid_arrive(cc, xgo);     // #8l+6
      epilogue_phase(p, cc, ec, cta, 3, l);
      if (sched[3].n == 0) grid_wait(cc, 8 * l + 7);  // (see grid_arrive: no arrival at #k+1 before #k is complete)
      grid_arrive(cc, 0, 0, 0, false);       // #8l+7 (split-K partials: read with ld.global.cg, no TMA consumer)
    }
    grid_wait(cc, 8 * p.L);
    ln_phase(p, cc, cta, false, 3, p.layers[p.L - 1].b_fc2, p.lnf_g, p.lnf_b);
    grid_arrive(cc, 0, 0, 0, false);         // #8L: exit barrier; CTA 0 re-arms the counter for the next launch
    if (cta == 0 && cc.ct == 0) {
      poll_counter(p.sync, static_cast<unsigned>(8 * p.L + 1) * ncta);
      *reinterpret_cast<volatile unsigned*>(p.sync) = 0u;
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 3) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc<512>(tmem_base);
  }
}

}  // namespace

size_t mega_plan(MegaState& m, int d, int ff, int ncta) {
  const int rows[4] = {3 * d, d, ff, d};
  const int ks[4] = {d, d, d, ff};
  m.ncta = ncta;
  m.h_tbl.clear();
  size_t ws_per_row = 0;
  for (int k = 0; k < 4; ++k) {
    MegaGemmShape& g = m.g[k];
    g.rows_out = rows[k];
    g.kb = ks[k] / 64;
    g.tiles = (rows[k] + 127) / 128;
    g.units = g.tiles * g.kb;
    g.tbl_off = static_cast<int>(m.h_tbl.size());
    int max_slots = 1;
    for (int t = 0; t < g.tiles; ++t) {
      // contributors of tile t: CTAs whose range [c*U/n, (c+1)*U/n) intersects [t*kb, (t+1)*kb)
      int first = -1, last = -1;
      const int nc = g.units < ncta ? g.units : ncta;  // CTAs taking part in this kind (see KindSched setup in the kernel)
      for (int c = 0; c < nc; ++c) {
        const long long u0 = static_cast<long long>(c) * g.units / nc, u1 = static_cast<long long>(c + 1) * g.units / nc;
        if (u0 < static_cast<long long>(t + 1) * g.kb && u1 > static_cast<long long>(t) * g.kb) {
          if (first < 0) first = c;
          last = c;
        }
      }
      const int ns = last - first + 1;
      if (ns > max_slots) max_slots = ns;
      m.h_tbl.push_back(static_cast<uint32_t>(first) | (static_cast<uint32_t>(ns) << 16));
    }
    const size_t need = static_cast<size_t>(max_slots) * g.rows_out;
    if (need > ws_per_row) ws_per_row = need;
  }
  m.tbl_entries = static_cast<int>(m.h_tbl.size());
  m.ws_floats_per_row = ws_per_row;
  return ws_per_row;
}

int mega_init() {
  cudaError_t e = cudaFuncSetAttribute(decode_mega_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  return e == cudaSuccess ? 0 : static_cast<int>(e);
}

int mega_launch(const MegaParams& p_in, cudaStream_t s) {
  MegaParams p = p_in;
  if (p.tbl_entries > kTblMax || p.d > 4096 || p.d % 8 || p.N > 256 || p.N % 16 || p.R > p.N) return static_cast<int>(cudaErrorInvalidValue);
  // shared memory budget: W ring + X ring (doubles as the vector phases' scratch) + strips / tables / barriers
  const int total = 227 * 1024 - 1024 /*alignment*/;
  const int xstage = p.N * 128;
  const int fixed = kAttnWarps * 192 * 4 + 64 + 64 + kTblMax * 4 + 512;
  // ring slots are handed over in pairs (two units per full / empty barrier) while at least two X pairs fit; at
  // 256 rows (32 KB activation tiles) the X ring holds three single tiles and every unit is handed over on its own
  p.nX = p.N <= 64 ? 8 : p.N <= 128 ? 4 : 3;
  p.grp = p.nX >= 4 ? 2 : 1;
  p.xring_bytes = p.nX * xstage > kVecScratch ? p.nX * xstage : kVecScratch;
  p.nW = (total - fixed - p.xring_bytes) / kWStage;
  if (p.nW > 12) p.nW = 12;
  if (p.grp == 2) p.nW &= ~1;
  if (p.nW < 2) return static_cast<int>(cudaErrorInvalidValue);
  p.nbar = 8 * p.L;
  const size_t smem = static_cast<size_t>(p.nW) * kWStage + p.xring_bytes + fixed + 1024;

  CUtensorMap mx, ma, mm;
  if (gemm_make_tmap(&mx, p.x, p.R, p.d, p.d, p.N)) return -1;
  if (gemm_make_tmap(&ma, p.att, p.R, p.d, p.d, p.N)) return -1;
  if (gemm_make_tmap(&mm, p.mlp, p.R, p.ff, p.ff, p.N)) return -1;

  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(p.ncta);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeCooperative;  // all CTAs co-resident: they wait on one another
  attr[0].val.cooperative = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, decode_mega_kernel, mx, ma, mm, p);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return static_cast<int>(e);
  }
  return 0;
}

}  // namespace ccb
