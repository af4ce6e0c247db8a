// Long-sequence prefill attention on tcgen05: softmax(Q K^T * scale) V for S > 256 (ViT-L/14: 257 tokens, ViT-L/14@336px:
// 577, the all-features mapper over either tower: 257 / 577 + prefix), non-causal, no key mask, no cache, no rotary,
// head_dim a multiple of 8 up to 256.  Same layout as attention_prefill: qkv [B*S, 3*H*hd] bf16 in, out [B*S, H*hd] out.
//
// One CTA of four warps per (128-query tile, head, image); thread t owns query row t = TMEM lane t.
//  * Q is staged once; K and V tiles of 64 keys go through a ring of NST stages with cp.async (16-byte chunks, zero-filled
//    past S and past head_dim), all as 128B-swizzled [rows][64 dims] blocks -- the layout a TMA box {64, rows} writes.
//    K is the K-major B operand of Q K^T; the very same V block is the MN-major B operand of P V (N = dims, K = keys), so
//    nothing is transposed.
//  * warp 0 (converged, one elected lane) issues S = Q K^T (M 128, N 64) into TMEM columns [0, 64) and O += P V (M 128,
//    N = HDP) into columns [64, 64 + HDP).
//  * softmax (online, base 2): each thread reads its 64 scores with tcgen05.ld, keeps the running max / sum in registers,
//    writes P = exp2(s - m) as ONE bf16 term into a swizzled K-major tile, and, when a row maximum of its warp grew,
//    rescales its O row in TMEM (tcgen05.ld -> * alpha -> tcgen05.st) once the previous P V has completed.  The exp of a
//    tile overlaps the previous tile's P V; the loads of tile j + NST - 1 overlap tile j's softmax.
//  * tail keys are masked to -inf; tail query rows are computed on zeros and not stored.  The summation order is fixed:
//    repeated calls are bit-identical.
#include "common.cuh"
#include "internal.h"
#include "ptx.cuh"

namespace ccb {

namespace {

constexpr int kLongThreads = 128;
constexpr int kLongKeys = 64;            // keys per tile (= one 128-byte swizzle row of P)

template <int HDP, int NST>
struct LongAttnCfg {
  static constexpr int QC = (HDP + 63) / 64;              // 64-dim blocks of Q / K / V
  static constexpr int kQBytes = QC * 128 * 128;
  static constexpr int kPBytes = 128 * 128;
  static constexpr int kKVBlock = kLongKeys * 128;        // one [64 keys][64 dims] block
  static constexpr int kStageBytes = 2 * QC * kKVBlock;   // K blocks then V blocks
  static constexpr int kBarOff = kQBytes + kPBytes + NST * kStageBytes;
  static constexpr int kSmem = kBarOff + 64 + 1024;       // + barriers / TMEM slot + alignment slack
  static constexpr int kTmemCols = (64 + HDP) <= 128 ? 128 : (64 + HDP) <= 256 ? 256 : 512;
};

__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src, uint32_t nbytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(nbytes) : "memory");
}
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }

template <int HDP, int NST>
__global__ void __launch_bounds__(kLongThreads, 1) attention_prefill_long_kernel(const bf16* __restrict__ qkv,
                                                                                bf16* __restrict__ out, int S, int H,
                                                                                int hd, float scale_log2) {
  using Cfg = LongAttnCfg<HDP, NST>;
  constexpr int QC = Cfg::QC, CPR = HDP / 8;   // 16-byte chunks per staged row
  extern __shared__ uint8_t long_smem[];
  const uint32_t raw = ptx::smem_u32(long_smem);
  const uint32_t sb = (raw + 1023u) & ~1023u;
  const uint32_t q_s = sb, p_s = sb + Cfg::kQBytes, kv_s = p_s + Cfg::kPBytes;
  const uint32_t bar_s = sb + Cfg::kBarOff, bar_o = bar_s + 8, slot = bar_s + 16;
  volatile uint32_t* slot_ptr = reinterpret_cast<volatile uint32_t*>(long_smem + (sb - raw) + Cfg::kBarOff + 16);
  const int tid = threadIdx.x, warp = tid >> 5;
  const int q0 = blockIdx.x * 128, h = blockIdx.y, b = blockIdx.z;
  const int d = H * hd;
  const long long ld = 3LL * d;
  const bf16* base = qkv + static_cast<size_t>(b) * S * ld + h * hd;
  const int n_tiles = (S + kLongKeys - 1) / kLongKeys;

  if (tid == 0) {
    ptx::mbar_init(bar_s, 1);
    ptx::mbar_init(bar_o, 1);
    ptx::fence_mbar_init();
  }
  if (warp == 0) ptx::tmem_alloc<Cfg::kTmemCols>(slot);
  ptx::grid_dep_wait();     // qkv comes from the c_attn GEMM this kernel is chained behind (PDL)
  ptx::grid_dep_launch();

  // chunk (row j, c) of a [rows][HDP] operand -> block c / 8, row j, 16-byte slot (c % 8) ^ (j % 8)
  auto sw_off = [](int j, int c, int block_bytes) -> uint32_t {
    return static_cast<uint32_t>((c >> 3) * block_bytes + j * 128 + (((c & 7) ^ (j & 7)) << 4));
  };
  auto load_tile = [&](int t) {
    const uint32_t st = kv_s + static_cast<uint32_t>((t % NST) * Cfg::kStageBytes);
    const int key0 = t * kLongKeys;
    for (int idx = tid; idx < kLongKeys * CPR; idx += kLongThreads) {
      const int j = idx / CPR, c = idx - j * CPR;
      const bool ok = key0 + j < S && c * 8 < hd;
      const bf16* src = ok ? base + (key0 + j) * ld + c * 8 : base;
      const uint32_t off = sw_off(j, c, Cfg::kKVBlock);
      cp_async16(st + off, ok ? src + d : base, ok ? 16u : 0u);
      cp_async16(st + QC * Cfg::kKVBlock + off, ok ? src + 2 * d : base, ok ? 16u : 0u);
    }
  };
  for (int idx = tid; idx < 128 * CPR; idx += kLongThreads) {
    const int j = idx / CPR, c = idx - j * CPR;
    const bool ok = q0 + j < S && c * 8 < hd;
    cp_async16(q_s + sw_off(j, c, 128 * 128), ok ? base + (q0 + j) * ld + c * 8 : base, ok ? 16u : 0u);
  }
#pragma unroll
  for (int t = 0; t < NST - 1; ++t) {
    if (t < n_tiles) load_tile(t);
    cp_async_commit();
  }
  cp_async_wait<NST - 2>();   // Q and tile 0
  ptx::fence_proxy_async();   // cp.async (generic proxy) writes -> tcgen05.mma reads
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem = *slot_ptr;
  const uint32_t tmem_o = tmem + 64u;
  const uint32_t lane_base = static_cast<uint32_t>(warp * 32) << 16;
  constexpr uint32_t idesc_s = ptx::umma_idesc_bf16(128, kLongKeys);
  constexpr uint32_t idesc_o = ptx::umma_idesc_bf16(128, HDP) | (1u << 16);   // B (V) MN-major

  auto issue_s = [&](int t) {   // S = Q K_t^T
    const uint32_t k_s = kv_s + static_cast<uint32_t>((t % NST) * Cfg::kStageBytes);
#pragma unroll
    for (int ks = 0; ks < HDP / 16; ++ks) {
      const uint64_t ad = ptx::umma_desc_k_sw128(q_s + (ks >> 2) * (128 * 128)) + 2u * (ks & 3);
      const uint64_t bd = ptx::umma_desc_k_sw128(k_s + (ks >> 2) * Cfg::kKVBlock) + 2u * (ks & 3);
      ptx::umma_bf16(tmem, ad, bd, idesc_s, ks > 0 ? 1u : 0u);
    }
    ptx::umma_commit(bar_s);
  };
  if (warp == 0 && ptx::elect_one()) issue_s(0);

  float m_run = -INFINITY, l_run = 0.f;
  for (int j = 0; j < n_tiles; ++j) {
    ptx::mbar_wait(bar_s, j & 1);
    ptx::tc_fence_after();
    float p[kLongKeys];
    {
      uint32_t r0[32], r1[32];
      ptx::tmem_ld32(tmem + lane_base, r0);
      ptx::tmem_ld32(tmem + lane_base + 32u, r1);
      ptx::tmem_ld_wait();
      const int valid = S - j * kLongKeys;   // keys of this tile that exist (>= 1)
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        p[i] = i < valid ? __uint_as_float(r0[i]) * scale_log2 : -INFINITY;
        p[32 + i] = 32 + i < valid ? __uint_as_float(r1[i]) * scale_log2 : -INFINITY;
      }
    }
    float mt = p[0];
#pragma unroll
    for (int i = 1; i < kLongKeys; ++i) mt = fmaxf(mt, p[i]);
    const float m_new = fmaxf(m_run, mt);
    float sum = 0.f;
#pragma unroll
    for (int i = 0; i < kLongKeys; ++i) {
      p[i] = ex2(p[i] - m_new);
      sum += p[i];
    }
    const float alpha = ex2(m_run - m_new);   // 0 on the first tile
    l_run = l_run * alpha + sum;
    const bool grew = m_new > m_run;
    m_run = m_new;

    // P V of the previous tile has completed: its stage, the P tile and O are free
    if (j > 0) {
      ptx::mbar_wait(bar_o, (j - 1) & 1);
      ptx::tc_fence_after();
    }
    if (j + NST - 1 < n_tiles) load_tile(j + NST - 1);
    cp_async_commit();
    if (j > 0 && __any_sync(0xffffffffu, grew)) {   // tcgen05.ld / st are warp-wide: rows that did not grow scale by 1
#pragma unroll 1
      for (int c = 0; c < HDP; c += 16) {
        uint32_t o[16];
        ptx::tmem_ld16(tmem_o + lane_base + c, o);
        ptx::tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 16; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * alpha);
        ptx::tmem_st16(tmem_o + lane_base + c, o);
      }
      ptx::tmem_st_wait();
    }
    {
      const uint32_t roff = p_s + static_cast<uint32_t>(tid) * 128u;
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const uint4 v = make_uint4(pack_bf16x2(p[8 * c], p[8 * c + 1]), pack_bf16x2(p[8 * c + 2], p[8 * c + 3]),
                                   pack_bf16x2(p[8 * c + 4], p[8 * c + 5]), pack_bf16x2(p[8 * c + 6], p[8 * c + 7]));
        asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(roff + ((c ^ (tid & 7)) << 4)), "r"(v.x), "r"(v.y),
                     "r"(v.z), "r"(v.w)
                     : "memory");
      }
    }
    cp_async_wait<NST - 2>();   // tile j + 1 has landed (this thread's chunks)
    ptx::fence_proxy_async();
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    if (warp == 0 && ptx::elect_one()) {
      if (j + 1 < n_tiles) issue_s(j + 1);
      const uint32_t v_s = kv_s + static_cast<uint32_t>((j % NST) * Cfg::kStageBytes + QC * Cfg::kKVBlock);
#pragma unroll
      for (int k = 0; k < kLongKeys / 16; ++k) {
        const uint64_t ad = ptx::umma_desc_k_sw128(p_s) + 2u * k;
        const uint64_t bd = ptx::umma_desc_mn_sw128(v_s + k * 2048, Cfg::kKVBlock);
        ptx::umma_bf16(tmem_o, ad, bd, idesc_o, (j > 0 || k > 0) ? 1u : 0u);
      }
      ptx::umma_commit(bar_o);
    }
  }

  ptx::mbar_wait(bar_o, (n_tiles - 1) & 1);
  ptx::tc_fence_after();
  const int row = q0 + tid;
  const float inv = 1.f / l_run;
  bf16* orow = out + (static_cast<size_t>(b) * S + row) * d + h * hd;
#pragma unroll 1
  for (int c = 0; c < HDP; c += 16) {
    uint32_t o[16];
    ptx::tmem_ld16(tmem_o + lane_base + c, o);
    ptx::tmem_ld_wait();
    if (row < S) {
#pragma unroll
      for (int hlf = 0; hlf < 2; ++hlf) {
        if (c + 8 * hlf < hd) {
          const uint32_t* src = o + 8 * hlf;
          uint4 pk;
          pk.x = pack_bf16x2(__uint_as_float(src[0]) * inv, __uint_as_float(src[1]) * inv);
          pk.y = pack_bf16x2(__uint_as_float(src[2]) * inv, __uint_as_float(src[3]) * inv);
          pk.z = pack_bf16x2(__uint_as_float(src[4]) * inv, __uint_as_float(src[5]) * inv);
          pk.w = pack_bf16x2(__uint_as_float(src[6]) * inv, __uint_as_float(src[7]) * inv);
          *reinterpret_cast<uint4*>(orow + c + 8 * hlf) = pk;
        }
      }
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc<Cfg::kTmemCols>(tmem);
  }
}

template <int HDP, int NST>
int launch_long(const bf16* qkv, bf16* out, int B, int S, int H, int hd, float scale, cudaStream_t s) {
  constexpr int smem = LongAttnCfg<HDP, NST>::kSmem;
  static bool configured_dev[kMaxDevices] = {};
  bool& configured = configured_dev[current_device_slot()];
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(attention_prefill_long_kernel<HDP, NST>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return (int)e;
    configured = true;
  }
  const float scale_log2 = scale * 1.4426950408889634f;
  cudaError_t e = launch_kernel(attention_prefill_long_kernel<HDP, NST>, dim3((S + 127) / 128, H, B), dim3(kLongThreads), smem, s,
                                true, qkv, out, S, H, hd, scale_log2);
  return e == cudaSuccess ? 0 : (int)e;
}

}  // namespace

int attention_prefill_long(const bf16* qkv, bf16* out, int B, int S, int H, int hd, float scale, cudaStream_t s) {
  if (B <= 0 || S <= 0) return 0;
  if (hd <= 0 || hd % 8 || hd > 256 || H <= 0) return (int)cudaErrorInvalidValue;
  // head_dim is padded to the next accumulator width the kernel is built for (the pad dims are zero-filled)
  if (hd <= 64) return launch_long<64, 3>(qkv, out, B, S, H, hd, scale, s);
  if (hd <= 96) return launch_long<96, 2>(qkv, out, B, S, H, hd, scale, s);
  if (hd <= 128) return launch_long<128, 2>(qkv, out, B, S, H, hd, scale, s);
  if (hd <= 160) return launch_long<160, 2>(qkv, out, B, S, H, hd, scale, s);
  if (hd <= 208) return launch_long<208, 2>(qkv, out, B, S, H, hd, scale, s);
  return launch_long<256, 2>(qkv, out, B, S, H, hd, scale, s);
}

}  // namespace ccb
