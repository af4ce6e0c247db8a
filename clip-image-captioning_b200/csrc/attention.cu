// Attention kernels.
//  * attention_prefill: full attention over a short sequence (S <= 256) for one (batch, head) per CTA.  Serves
//    the ViT (S=50, hd=64, non-causal), the prefix mapper (S=clip_len+P, hd=d/8, non-causal; reference
//    layers/MultiHeadAttention.py:24-41) and the LM prefill (causal; HF GPT2Attention / GPTJAttention), where
//    it also writes K/V into the paged cache.  S > 256 (ViT-L towers, the all-features mapper over them) is handed to the
//    tcgen05 kernel of attention_long.cu.
//  * attention_decode: one query token per row against the paged KV cache; memory-bound, 16-byte loads,
//    online softmax, 4 warps per (row, head) each striding over the context, merged through shared memory.
#include <stdlib.h>

#include "common.cuh"
#include "internal.h"
#include "ptx.cuh"

namespace ccb {

namespace {

__device__ __forceinline__ size_t kv_index(const KvCache& c, int layer, int kv, int page, int h, int t) {
  return ((((static_cast<size_t>(layer) * 2 + kv) * c.num_pages + page) * c.H + h) * c.page_tokens + t) * c.hd;
}

// GPT-J rotary ("rotate_every_two", HF modeling_gptj.py:47-67): pairs (2i, 2i+1) of the first rotary_dim dims.
__device__ __forceinline__ void rotary_pair(float& a, float& b, int pair_idx, int pos, int rotary_dim) {
  const float inv_freq = powf(10000.f, -2.f * pair_idx / rotary_dim);
  float sn, cs;
  sincosf(pos * inv_freq, &sn, &cs);
  const float a2 = a * cs - b * sn;
  const float b2 = b * cs + a * sn;
  a = a2;
  b = b2;
}

// ------------------------------------------------------------------------------------------------ prefill
// smem: Ks [S][hd/2+1] words (bf16x2, padded -> conflict-free column walks), Vs [S][hd/2] words,
//       per-warp q row (hd floats) and probability row (S floats).
constexpr int kPrefillWarps = 8;

__global__ void __launch_bounds__(kPrefillWarps * 32) attention_prefill_kernel(
    const bf16* __restrict__ qkv, bf16* __restrict__ out, int S, int H, int hd, float scale, int causal,
    KvCache cache, int layer, const int* __restrict__ block_table, int pos0, int rotary_dim, int write_cache,
    const uint8_t* __restrict__ key_mask) {
  extern __shared__ uint32_t smem_u[];
  const int h = blockIdx.x, b = blockIdx.y;
  const int d = H * hd;
  const int hw = hd / 2;        // words per row
  const int kstride = hw + 1;
  uint32_t* Ks = smem_u;
  uint32_t* Vs = Ks + S * kstride;
  // q rows are read back as float2: keep the fp32 region 8-byte aligned (S * (2 * hw + 1) words can be odd)
  float* qbuf = reinterpret_cast<float*>(smem_u + ((S * (kstride + hw) + 1) & ~1));  // [warps][hd]
  float* pbuf = qbuf + kPrefillWarps * hd;                        // [warps][S]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const bf16* base = qkv + static_cast<size_t>(b) * S * 3 * d;

  // stage K and V of this head (bf16 pairs); apply rotary to K first when requested
  for (int idx = threadIdx.x; idx < S * hw; idx += blockDim.x) {
    const int j = idx / hw, w = idx % hw;
    const bf16* rowp = base + static_cast<size_t>(j) * 3 * d;
    uint32_t kw = *reinterpret_cast<const uint32_t*>(rowp + d + h * hd + 2 * w);
    const uint32_t vw = *reinterpret_cast<const uint32_t*>(rowp + 2 * d + h * hd + 2 * w);
    if (rotary_dim > 0 && 2 * w < rotary_dim) {
      float2 kf = unpack_bf16x2(kw);
      rotary_pair(kf.x, kf.y, w, pos0 + j, rotary_dim);
      kw = pack_bf16x2(kf.x, kf.y);
    }
    Ks[j * kstride + w] = kw;
    Vs[j * hw + w] = vw;
    if (write_cache) {
      const int pos = pos0 + j;
      const int page = block_table[static_cast<size_t>(b) * cache.max_pages_per_row + pos / cache.page_tokens];
      const int t = pos % cache.page_tokens;
      *reinterpret_cast<uint32_t*>(cache.base + kv_index(cache, layer, 0, page, h, t) + 2 * w) = kw;
      *reinterpret_cast<uint32_t*>(cache.base + kv_index(cache, layer, 1, page, h, t) + 2 * w) = vw;
    }
  }
  __syncthreads();

  float* myq = qbuf + warp * hd;
  float* myp = pbuf + warp * S;
  for (int i = warp; i < S; i += kPrefillWarps) {
    // q row -> fp32 in shared (rotary applied)
    const bf16* qrow = base + static_cast<size_t>(i) * 3 * d + h * hd;
    for (int w = lane; w < hw; w += 32) {
      float2 qf = unpack_bf16x2(*reinterpret_cast<const uint32_t*>(qrow + 2 * w));
      if (rotary_dim > 0 && 2 * w < rotary_dim) rotary_pair(qf.x, qf.y, w, pos0 + i, rotary_dim);
      myq[2 * w] = qf.x;
      myq[2 * w + 1] = qf.y;
    }
    __syncwarp();
    const int jmax = causal ? i + 1 : S;  // keys [0, jmax)
    float sc[8];
    float mx = -INFINITY;
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      const int j = c * 32 + lane;
      float acc = -INFINITY;
      if (c * 32 < jmax && j < jmax && (key_mask == nullptr || key_mask[static_cast<size_t>(b) * S + j])) {
        acc = 0.f;
        const uint32_t* kr = Ks + j * kstride;
        for (int w = 0; w < hw; ++w) {
          const float2 kf = unpack_bf16x2(kr[w]);
          const float2 qf = *reinterpret_cast<const float2*>(myq + 2 * w);
          acc = fmaf(qf.x, kf.x, acc);
          acc = fmaf(qf.y, kf.y, acc);
        }
        acc *= scale;
      }
      sc[c] = acc;
      mx = fmaxf(mx, acc);
    }
    mx = warp_max(mx);
    float sum = 0.f;
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      const float e = (sc[c] == -INFINITY) ? 0.f : expf(sc[c] - mx);
      sc[c] = e;
      sum += e;
    }
    sum = warp_sum(sum);
    const float inv = sum > 0.f ? 1.f / sum : 0.f;
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      const int j = c * 32 + lane;
      if (j < jmax) myp[j] = sc[c] * inv;
    }
    __syncwarp();
    bf16* orow = out + (static_cast<size_t>(b) * S + i) * d + h * hd;
    for (int w = lane; w < hw; w += 32) {
      float a0 = 0.f, a1 = 0.f;
      for (int j = 0; j < jmax; ++j) {
        const float p = myp[j];
        const float2 vf = unpack_bf16x2(Vs[j * hw + w]);
        a0 = fmaf(p, vf.x, a0);
        a1 = fmaf(p, vf.y, a1);
      }
      *reinterpret_cast<uint32_t*>(orow + 2 * w) = pack_bf16x2(a0, a1);
    }
    __syncwarp();
  }
}

// ------------------------------------------------------------------------------------------------ prefill, tensor cores
// Same operator for S <= 128, head_dim % 8 == 0, head_dim <= 256, no rotary: one CTA per (batch, head), one warp per
// 16 query rows, mma.sync m16n8k16 (bf16 in, fp32 accumulate) for Q K^T and P V.  K and V of the head are staged once
// in shared memory (row pitch head_dim rounded to 16, + 8 elements: conflict-free fragment loads and 16-byte aligned
// ldmatrix rows); the scores of a query tile stay in registers from Q K^T through the softmax into the P operand.  The scalar kernel above spent
// ~4000 instructions per warp on this (88 us per GPT2-XL layer at batch 64); this one is a few hundred.
__device__ __forceinline__ void mma_bf16_16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void ldmatrix_x2_trans(uint32_t& r0, uint32_t& r1, uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x2.trans.shared.b16 {%0,%1}, [%2];" : "=r"(r0), "=r"(r1) : "r"(addr));
}

// OVL: K and V share ONE staging buffer (V is requested once every warp has its scores in registers): half the shared memory,
// twice the CTAs per SM -- the mapper's 80 keys x head_dim 200 (69 KB for both) ran 512 CTAs on 444 slots, i.e. in two waves.
// Only without rotary / cache append (the host picks it for the mapper shapes).
template <int NT, int KS, bool OVL = false>   // NT: key tiles of 8 (even, >= 2 * warps); KS: head_dim steps of 16
__global__ void __launch_bounds__(256) attention_prefill_mma_kernel(
    const bf16* __restrict__ qkv, bf16* __restrict__ out, int S, int H, int hd, float scale, int causal,
    KvCache cache, int layer, const int* __restrict__ block_table, int pos0, int write_cache,
    const uint8_t* __restrict__ key_mask, int rotary_dim) {
  extern __shared__ uint4 smem_u4[];
  const int h = blockIdx.x, b = blockIdx.y;
  const int d = H * hd;
  const int HDP = KS * 16 + 8;            // row pitch in elements
  const int S16 = NT * 8;                 // staged key rows
  bf16* Ks = reinterpret_cast<bf16*>(smem_u4);
  bf16* Vs = OVL ? Ks : Ks + S16 * HDP;
  float* mask_add = reinterpret_cast<float*>(Vs + S16 * HDP);   // 0 or -inf per key
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  const bf16* base = qkv + static_cast<size_t>(b) * S * 3 * d;
  ptx::grid_dep_wait();     // qkv comes from the c_attn GEMM this kernel is chained behind (PDL)
  ptx::grid_dep_launch();

  // ---- stage K / V (16-byte chunks, zero padded), append them to the KV cache, build the key mask.
  // Every chunk is requested with cp.async before the first one is used: a loop of load -> store per chunk has one
  // L2 round trip per iteration on its critical path (the mapper's 80 x 27 chunks on 160 threads: 14 of them).
  const int cpr = HDP / 8;                // chunks per staged row
  {
    const uint32_t ks_u32 = ptx::smem_u32(Ks), vs_u32 = ptx::smem_u32(Vs);
    for (int idx = threadIdx.x; idx < S16 * cpr; idx += blockDim.x) {
      const int j = idx / cpr, c = idx - j * cpr;
      const bool ok = j < S && c * 8 < hd;
      const bf16* rowp = ok ? base + static_cast<size_t>(j) * 3 * d + h * hd + c * 8 : base;
      const uint32_t off = static_cast<uint32_t>((j * HDP + c * 8) * 2);
      const uint32_t nbytes = ok ? 16u : 0u;   // 0: the chunk is zero-filled
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(ks_u32 + off), "l"(rowp + (ok ? d : 0)), "r"(nbytes) : "memory");
      if constexpr (!OVL)
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(vs_u32 + off), "l"(rowp + (ok ? 2 * d : 0)), "r"(nbytes) : "memory");
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
    asm volatile("cp.async.wait_group 0;" ::: "memory");
  }
  if (rotary_dim > 0 || write_cache) {
    // (each thread revisits the chunks it requested itself: its own cp.async writes are visible to it after the wait)
    for (int idx = threadIdx.x; idx < S16 * cpr; idx += blockDim.x) {
      const int j = idx / cpr, c = idx - j * cpr;
      if (!(j < S && c * 8 < hd)) continue;
      uint4 kk = *reinterpret_cast<const uint4*>(Ks + j * HDP + c * 8);
      if (c * 8 < rotary_dim) {   // GPT-J rotary on the first rotary_dim dims of K (pairs 2i, 2i+1), rounded to bf16 as cached
        uint32_t* kw = reinterpret_cast<uint32_t*>(&kk);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          if (c * 8 + 2 * e < rotary_dim) {
            float2 kf = unpack_bf16x2(kw[e]);
            rotary_pair(kf.x, kf.y, c * 4 + e, pos0 + j, rotary_dim);
            kw[e] = pack_bf16x2(kf.x, kf.y);
          }
        }
        *reinterpret_cast<uint4*>(Ks + j * HDP + c * 8) = kk;
      }
      if (write_cache) {
        const uint4 vv = *reinterpret_cast<const uint4*>(Vs + j * HDP + c * 8);
        const int pos = pos0 + j;
        const int page = block_table[static_cast<size_t>(b) * cache.max_pages_per_row + pos / cache.page_tokens];
        const int tin = pos % cache.page_tokens;
        *reinterpret_cast<uint4*>(cache.base + kv_index(cache, layer, 0, page, h, tin) + c * 8) = kk;
        *reinterpret_cast<uint4*>(cache.base + kv_index(cache, layer, 1, page, h, tin) + c * 8) = vv;
      }
    }
  }
  for (int j = threadIdx.x; j < S16; j += blockDim.x)
    mask_add[j] = (j < S && (key_mask == nullptr || key_mask[static_cast<size_t>(b) * S + j])) ? 0.f : -INFINITY;
  __syncthreads();

  const int r0 = warp * 16;               // this warp's query rows r0 + g, r0 + g + 8
  if (!OVL && r0 >= S) return;            // (the launch has ceil(S / 16) warps: never taken; OVL has barriers below)
  const int row_a = r0 + g, row_b = r0 + g + 8;

  // ---- Q fragments straight from global memory (A operand, row-major), scores = Q K^T
  constexpr bool kStreamQ = KS > 16;   // head_dim 512 (the 4096-wide mapper): KS x 4 fragment registers do not fit
  const bf16* qa = base + static_cast<size_t>(row_a) * 3 * d + h * hd;
  const bf16* qb = base + static_cast<size_t>(row_b) * 3 * d + h * hd;
  auto load_q = [&](int ks, uint32_t (&f)[4]) {
    const int k0 = ks * 16 + 2 * t, k1 = k0 + 8;
    f[0] = (row_a < S && k0 < hd) ? *reinterpret_cast<const uint32_t*>(qa + k0) : 0u;
    f[1] = (row_b < S && k0 < hd) ? *reinterpret_cast<const uint32_t*>(qb + k0) : 0u;
    f[2] = (row_a < S && k1 < hd) ? *reinterpret_cast<const uint32_t*>(qa + k1) : 0u;
    f[3] = (row_b < S && k1 < hd) ? *reinterpret_cast<const uint32_t*>(qb + k1) : 0u;
  };
  float sc[NT][4];
#pragma unroll
  for (int nt = 0; nt < NT; ++nt) sc[nt][0] = sc[nt][1] = sc[nt][2] = sc[nt][3] = 0.f;
  if constexpr (!kStreamQ) {
    uint32_t qf[KS][4];
#pragma unroll
    for (int ks = 0; ks < KS; ++ks) {
      load_q(ks, qf[ks]);
      if (ks * 16 < rotary_dim) {   // rotary on q (the MMA operand is bf16: the rotated pair is rounded once more)
        const int k0 = ks * 16 + 2 * t, k1 = k0 + 8;
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int k = (e < 2) ? k0 : k1;
          const int row = (e & 1) ? row_b : row_a;
          if (k < rotary_dim && row < S) {
            float2 f = unpack_bf16x2(qf[ks][e]);
            rotary_pair(f.x, f.y, k >> 1, pos0 + row, rotary_dim);
            qf[ks][e] = pack_bf16x2(f.x, f.y);
          }
        }
      }
    }
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
      const bf16* krow = Ks + (nt * 8 + g) * HDP + 2 * t;
#pragma unroll
      for (int ks = 0; ks < KS; ++ks) {
        const uint32_t b0 = *reinterpret_cast<const uint32_t*>(krow + ks * 16);
        const uint32_t b1 = *reinterpret_cast<const uint32_t*>(krow + ks * 16 + 8);
        mma_bf16_16816(sc[nt], qf[ks], b0, b1);
      }
    }
  } else {
    // the scores accumulate head_dim step by step; the fragments of a step are requested four steps ahead (no rotary
    // on this path: the host sends rotary models to the variants above)
    uint32_t qr[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i) load_q(i, qr[i]);
#pragma unroll
    for (int ks = 0; ks < KS; ++ks) {
      uint32_t cur[4] = {qr[ks & 3][0], qr[ks & 3][1], qr[ks & 3][2], qr[ks & 3][3]};
      if (ks + 4 < KS) load_q(ks + 4, qr[ks & 3]);
#pragma unroll
      for (int nt = 0; nt < NT; ++nt) {
        const bf16* krow = Ks + (nt * 8 + g) * HDP + 2 * t;
        const uint32_t b0 = *reinterpret_cast<const uint32_t*>(krow + ks * 16);
        const uint32_t b1 = *reinterpret_cast<const uint32_t*>(krow + ks * 16 + 8);
        mma_bf16_16816(sc[nt], cur, b0, b1);
      }
    }
  }
  // ---- mask, softmax over the row (thread holds keys nt*8 + 2t, +1 of rows a and b; the 4 lanes of a quad share a row)
  float mx_a = -INFINITY, mx_b = -INFINITY;
#pragma unroll
  for (int nt = 0; nt < NT; ++nt) {
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int key = nt * 8 + 2 * t + e;
      const float m = mask_add[key];
      const float va = (causal && key > row_a) ? -INFINITY : sc[nt][e] * scale + m;
      const float vb = (causal && key > row_b) ? -INFINITY : sc[nt][2 + e] * scale + m;
      sc[nt][e] = va;
      sc[nt][2 + e] = vb;
      mx_a = fmaxf(mx_a, va);
      mx_b = fmaxf(mx_b, vb);
    }
  }
  mx_a = fmaxf(mx_a, __shfl_xor_sync(0xffffffffu, mx_a, 1));
  mx_a = fmaxf(mx_a, __shfl_xor_sync(0xffffffffu, mx_a, 2));
  mx_b = fmaxf(mx_b, __shfl_xor_sync(0xffffffffu, mx_b, 1));
  mx_b = fmaxf(mx_b, __shfl_xor_sync(0xffffffffu, mx_b, 2));
  float sum_a = 0.f, sum_b = 0.f;
#pragma unroll
  for (int nt = 0; nt < NT; ++nt) {
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const float pa = (sc[nt][e] == -INFINITY) ? 0.f : expf(sc[nt][e] - mx_a);
      const float pb = (sc[nt][2 + e] == -INFINITY) ? 0.f : expf(sc[nt][2 + e] - mx_b);
      sc[nt][e] = pa;
      sc[nt][2 + e] = pb;
      sum_a += pa;
      sum_b += pb;
    }
  }
  sum_a += __shfl_xor_sync(0xffffffffu, sum_a, 1);
  sum_a += __shfl_xor_sync(0xffffffffu, sum_a, 2);
  sum_b += __shfl_xor_sync(0xffffffffu, sum_b, 1);
  sum_b += __shfl_xor_sync(0xffffffffu, sum_b, 2);
  const float inv_a = sum_a > 0.f ? 1.f / sum_a : 0.f, inv_b = sum_b > 0.f ? 1.f / sum_b : 0.f;
  // ---- P as the A operand of the second product (keys are its k dimension: tile pair (2kk, 2kk+1) = 16 keys).
  // P is split into two bf16 terms (p = hi + lo, |lo| <= 2^-9 |p|) and multiplied in two MMAs, so the probabilities
  // keep ~16 significant bits: the result stays within fp32-accumulation noise of the fp32-softmax formulation and
  // greedy captions on near-tie logits do not depend on the kernel choice.
  uint32_t pf[NT / 2][4], pl[NT / 2][4];
#pragma unroll
  for (int kk = 0; kk < NT / 2; ++kk) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int nt = 2 * kk + (q >> 1), e = (q & 1) * 2;   // q: 0 -> (tile 2kk, row a), 1 -> (2kk, row b), 2 -> (2kk+1, a), 3 -> (2kk+1, b)
      const float inv = (q & 1) ? inv_b : inv_a;
      const float x0 = sc[nt][e] * inv, x1 = sc[nt][e + 1] * inv;
      const uint32_t hi = pack_bf16x2(x0, x1);
      const float2 hf = unpack_bf16x2(hi);
      pf[kk][q] = hi;
      pl[kk][q] = pack_bf16x2(x0 - hf.x, x1 - hf.y);
    }
  }
  if constexpr (OVL) {
    __syncthreads();   // every warp has read its K fragments: the buffer takes V now
    const uint32_t vdst = ptx::smem_u32(Vs);
    for (int idx = threadIdx.x; idx < S16 * cpr; idx += blockDim.x) {
      const int j = idx / cpr, c = idx - j * cpr;
      const bool ok = j < S && c * 8 < hd;
      const bf16* rowp = ok ? base + static_cast<size_t>(j) * 3 * d + h * hd + c * 8 + 2 * d : base;
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(vdst + static_cast<uint32_t>((j * HDP + c * 8) * 2)), "l"(rowp),
                   "r"(ok ? 16u : 0u) : "memory");
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncthreads();
  }
  // ---- O = P V, 64 output dims at a time
  const uint32_t vs_u32 = ptx::smem_u32(Vs);
  bf16* oa = out + (static_cast<size_t>(b) * S + row_a) * d + h * hd;
  bf16* ob = out + (static_cast<size_t>(b) * S + row_b) * d + h * hd;
#pragma unroll 1
  for (int dc = 0; dc < hd; dc += 64) {
    float o[8][4];
#pragma unroll
    for (int n = 0; n < 8; ++n) o[n][0] = o[n][1] = o[n][2] = o[n][3] = 0.f;
#pragma unroll
    for (int kk = 0; kk < NT / 2; ++kk) {
      // lanes 0..15 address the 16 key rows of this k step (lanes 16..31 repeat them: ignored by .x2)
      const uint32_t vrow = vs_u32 + static_cast<uint32_t>(((kk * 16 + (lane & 15)) * HDP + dc) * 2);
#pragma unroll
      for (int n = 0; n < 8; ++n) {
        if (dc + n * 8 < hd) {   // (warp-uniform)
          uint32_t b0, b1;
          ldmatrix_x2_trans(b0, b1, vrow + n * 16);
          mma_bf16_16816(o[n], pf[kk], b0, b1);
          mma_bf16_16816(o[n], pl[kk], b0, b1);
        }
      }
    }
#pragma unroll
    for (int n = 0; n < 8; ++n) {
      const int dim = dc + n * 8 + 2 * t;
      if (dim < hd) {
        if (row_a < S) *reinterpret_cast<uint32_t*>(oa + dim) = pack_bf16x2(o[n][0], o[n][1]);
        if (row_b < S) *reinterpret_cast<uint32_t*>(ob + dim) = pack_bf16x2(o[n][2], o[n][3]);
      }
    }
  }
}

template <int NT, int KS, bool OVL = false>
int launch_prefill_mma(const bf16* qkv, bf16* out, int B, int S, int H, int hd, float scale, int causal, const KvCache& c,
                       int layer, const int* block_table, int pos0, int write_cache, const uint8_t* key_mask, int rotary_dim,
                       cudaStream_t s) {
  const int HDP = KS * 16 + 8, S16 = NT * 8;
  const size_t smem = static_cast<size_t>(OVL ? 1 : 2) * S16 * HDP * sizeof(bf16) + S16 * sizeof(float);
  static size_t configured_dev[kMaxDevices] = {};
  size_t& configured = configured_dev[current_device_slot()];
  if (smem > 48 * 1024 && smem > configured) {
    cudaError_t e = cudaFuncSetAttribute(attention_prefill_mma_kernel<NT, KS, OVL>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (e != cudaSuccess) return (int)e;
    configured = smem;
  }
  const int warps = (S + 15) / 16;
  cudaError_t e = launch_kernel(attention_prefill_mma_kernel<NT, KS, OVL>, dim3(H, B), dim3(warps * 32), smem, s, true, qkv, out, S, H, hd,
                                scale, causal, c, layer, block_table, pos0, write_cache, key_mask, rotary_dim);
  return e == cudaSuccess ? 0 : (int)e;
}

// ---------------------------------------------------------------------------------------------------------------
// tcgen05 / TMEM prefill attention for head_dim 64 and S <= 64 (ViT-B/32: S = 50; GPT-2 prefill of a 40-token prefix).
// One CTA of four warps per (head, batch).  Q, K and V^T are staged by the threads as 128B-swizzled K-major tiles (what
// a TMA box {64, 64 rows} would write; V is transposed on the way so that P.V has its K dimension = keys contiguous);
// S = Q.K^T is ONE M = 64 x N = 64 accumulator in TMEM (4 tcgen05.mma of K = 16); the M = 64 accumulator keeps row
// 16 w + i in lane i of warp w's quadrant, so lanes 0-15 of every warp own one query row each and do the whole softmax
// in registers (no shuffles); P, normalised and split into bf16 hi + lo terms like the mma.sync kernel (same accuracy),
// goes back through shared memory as the A operand of O = P.V (8 tcgen05.mma into a second accumulator).
// K / V are appended to the paged cache while they are staged (write_cache), the HF key mask and the causal mask are
// applied to the scores.  Rotary models (GPT-J) keep the mma.sync kernel.
__device__ __forceinline__ void sts_u16(uint32_t addr, uint16_t v) {
  asm volatile("st.shared.u16 [%0], %1;" ::"r"(addr), "h"(v) : "memory");
}
__device__ __forceinline__ void sts_v4(uint32_t addr, uint4 v) {
  asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// Q / K / V^T tiles (P_hi / P_lo reuse Q / K once S is computed) + key mask + barrier / TMEM slot + alignment: 8 CTAs per SM
constexpr int kUmmaAttnSmem = 3 * 8192 + 64 * 4 + 64 + 1024;

__global__ void __launch_bounds__(128) attention_prefill_umma_kernel(
    const bf16* __restrict__ qkv, bf16* __restrict__ out, int S, int H, float scale, int causal, KvCache cache, int layer,
    const int* __restrict__ block_table, int pos0, int write_cache, const uint8_t* __restrict__ key_mask) {
  constexpr int HD = 64;
  extern __shared__ uint8_t umma_smem[];
  const uint32_t raw = ptx::smem_u32(umma_smem);
  const uint32_t sb = (raw + 1023u) & ~1023u;
  uint8_t* gen = umma_smem + (sb - raw);
  const uint32_t q_s = sb, k_s = sb + 8192, vt_s = sb + 16384, ph_s = q_s, pl_s = k_s;
  float* mask_add = reinterpret_cast<float*>(gen + 24576);
  const uint32_t bar = sb + 24576 + 256, slot = bar + 16;
  volatile uint32_t* slot_ptr = reinterpret_cast<volatile uint32_t*>(gen + 24576 + 256 + 16);
  const int h = blockIdx.x, b = blockIdx.y;
  const int d = H * HD;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (tid == 0) {
    ptx::mbar_init(bar, 1);
    ptx::fence_mbar_init();
  }
  if (warp == 0) ptx::tmem_alloc<64>(slot);   // S and, after the softmax has read it, O share the 64 columns
  ptx::grid_dep_wait();     // qkv comes from the c_attn GEMM this kernel is chained behind (PDL)
  ptx::grid_dep_launch();
  // ---- stage Q and K (row-major, swizzled), append K to the cache, key mask; then S = Q K^T is issued ...
  // All twelve 16-byte chunks of a thread (Q, K, V of its four (key, chunk) pairs) are requested before the first one is
  // stored: the shared-memory stores are asm volatile, so a load -> store loop would put one L2 round trip per iteration
  // (eight in all) on the critical path of a CTA that lives for a few microseconds.
  const bf16* base = qkv + static_cast<size_t>(b) * S * 3 * d + h * HD;
  const int* bt = block_table + static_cast<size_t>(b) * cache.max_pages_per_row;
  uint4 q4[4], k4[4], v4[4];
#pragma unroll
  for (int it = 0; it < 4; ++it) {
    const int idx = tid + it * 128;
    const int j = idx >> 3, c = idx & 7;
    q4[it] = k4[it] = v4[it] = make_uint4(0u, 0u, 0u, 0u);
    if (j < S) {
      const bf16* rowp = base + static_cast<size_t>(j) * 3 * d + c * 8;
      q4[it] = *reinterpret_cast<const uint4*>(rowp);
      k4[it] = *reinterpret_cast<const uint4*>(rowp + d);
      v4[it] = *reinterpret_cast<const uint4*>(rowp + 2 * d);
    }
  }
#pragma unroll
  for (int it = 0; it < 4; ++it) {
    const int idx = tid + it * 128;
    const int j = idx >> 3, c = idx & 7;
    if (j < S && write_cache) {
      const int pos = pos0 + j;
      *reinterpret_cast<uint4*>(cache.base + kv_index(cache, layer, 0, bt[pos / cache.page_tokens], h, pos % cache.page_tokens) + c * 8) = k4[it];
    }
    const uint32_t off = static_cast<uint32_t>(j) * 128u + (static_cast<uint32_t>(c ^ (j & 7)) << 4);
    sts_v4(q_s + off, q4[it]);
    sts_v4(k_s + off, k4[it]);
  }
  if (tid < 64) mask_add[tid] = (tid < S && (key_mask == nullptr || key_mask[static_cast<size_t>(b) * S + tid])) ? 0.f : -INFINITY;
  ptx::fence_proxy_async();          // generic stores -> tcgen05.mma (async proxy) reads
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem = *slot_ptr;
  const uint32_t idesc = ptx::umma_idesc_bf16(64, 64);
  if (warp == 0 && ptx::elect_one()) {
    const uint64_t ad = ptx::umma_desc_k_sw128(q_s), bd = ptx::umma_desc_k_sw128(k_s);
#pragma unroll
    for (int k = 0; k < 4; ++k) ptx::umma_bf16(tmem, ad + 2u * k, bd + 2u * k, idesc, k > 0 ? 1u : 0u);
    ptx::umma_commit(bar);
  }
  // ---- ... while V is transposed: element (dim n, key j) -> row n, 16-byte chunk (j / 8) ^ (n % 8), slot j % 8.  A lane's
  // eight elements are visited in an order rotated by its chunk index c, so that the eight lanes that share a key write
  // eight different rows AND chunks (no bank conflicts; the loads stay 128 contiguous bytes per key)
#pragma unroll
  for (int it = 0; it < 4; ++it) {
    const int idx = tid + it * 128;
    const int j = idx >> 3, c = idx & 7;
    const uint4 vv = v4[it];
    if (j < S && write_cache) {
      const int pos = pos0 + j;
      *reinterpret_cast<uint4*>(cache.base + kv_index(cache, layer, 1, bt[pos / cache.page_tokens], h, pos % cache.page_tokens) + c * 8) = vv;
    }
    const uint64_t lo64 = static_cast<uint64_t>(vv.x) | (static_cast<uint64_t>(vv.y) << 32);
    const uint64_t hi64 = static_cast<uint64_t>(vv.z) | (static_cast<uint64_t>(vv.w) << 32);
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int ee = (e + c) & 7, n = c * 8 + ee;
      const uint16_t val = static_cast<uint16_t>(((ee & 4) ? hi64 : lo64) >> (16 * (ee & 3)));
      sts_u16(vt_s + static_cast<uint32_t>(n) * 128u + (static_cast<uint32_t>((j >> 3) ^ (n & 7)) << 4) + static_cast<uint32_t>(j & 7) * 2u, val);
    }
  }
  ptx::mbar_wait(bar, 0);
  ptx::tc_fence_after();
  // ---- softmax: lanes 0-15 of each warp hold the 64 scores of row 16 warp + lane; lanes 16-31 take the upper 32 columns
  // of the same row over by shuffle, so that all 32 lanes work (half a row each)
  const int row = warp * 16 + (lane & 15);
  {
    uint32_t r0[32], r1[32];
    ptx::tmem_ld32(tmem + (static_cast<uint32_t>(warp * 32) << 16), r0);
    ptx::tmem_ld32(tmem + (static_cast<uint32_t>(warp * 32) << 16) + 32u, r1);
    ptx::tmem_ld_wait();
    const bool upper = lane >= 16;
    const int col0 = upper ? 32 : 0;
    float sc[32];
    float mx = -INFINITY;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const uint32_t hi_half = __shfl_sync(0xffffffffu, r1[j], lane & 15);
      const float raw_s = __uint_as_float(upper ? hi_half : r0[j]);
      const int key = col0 + j;
      const float v = (causal && key > row) ? -INFINITY : raw_s * scale + mask_add[key];
      sc[j] = v;
      mx = fmaxf(mx, v);
    }
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 16));
    float sum = 0.f;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const float pr = (sc[j] == -INFINITY) ? 0.f : expf(sc[j] - mx);
      sc[j] = pr;
      sum += pr;
    }
    sum += __shfl_xor_sync(0xffffffffu, sum, 16);
    const float inv = sum > 0.f ? 1.f / sum : 0.f;
    const uint32_t roff = static_cast<uint32_t>(row) * 128u;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      uint32_t hi[4], lo[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float x0 = sc[c * 8 + 2 * e] * inv, x1 = sc[c * 8 + 2 * e + 1] * inv;
        hi[e] = pack_bf16x2(x0, x1);
        const float2 hf = unpack_bf16x2(hi[e]);
        lo[e] = pack_bf16x2(x0 - hf.x, x1 - hf.y);
      }
      const uint32_t off = roff + (static_cast<uint32_t>(((upper ? 4 : 0) + c) ^ (row & 7)) << 4);
      sts_v4(ph_s + off, make_uint4(hi[0], hi[1], hi[2], hi[3]));
      sts_v4(pl_s + off, make_uint4(lo[0], lo[1], lo[2], lo[3]));
    }
  }
  ptx::fence_proxy_async();
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  // ---- O = P V (hi and lo terms into one accumulator)
  if (warp == 0 && ptx::elect_one()) {
    const uint64_t ah = ptx::umma_desc_k_sw128(ph_s), al = ptx::umma_desc_k_sw128(pl_s), bd = ptx::umma_desc_k_sw128(vt_s);
#pragma unroll
    for (int k = 0; k < 4; ++k) ptx::umma_bf16(tmem, ah + 2u * k, bd + 2u * k, idesc, k > 0 ? 1u : 0u);
#pragma unroll
    for (int k = 0; k < 4; ++k) ptx::umma_bf16(tmem, al + 2u * k, bd + 2u * k, idesc, 1u);
    ptx::umma_commit(bar);
  }
  ptx::mbar_wait(bar, 1);
  ptx::tc_fence_after();
  {
    uint32_t r0[32], r1[32];
    ptx::tmem_ld32(tmem + (static_cast<uint32_t>(warp * 32) << 16), r0);
    ptx::tmem_ld32(tmem + (static_cast<uint32_t>(warp * 32) << 16) + 32u, r1);
    ptx::tmem_ld_wait();
    if (lane < 16 && row < S) {
      bf16* op = out + (static_cast<size_t>(b) * S + row) * d + h * HD;
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        uint4 pk;
        const uint32_t* src = c < 4 ? r0 + c * 8 : r1 + (c - 4) * 8;
        pk.x = pack_bf16x2(__uint_as_float(src[0]), __uint_as_float(src[1]));
        pk.y = pack_bf16x2(__uint_as_float(src[2]), __uint_as_float(src[3]));
        pk.z = pack_bf16x2(__uint_as_float(src[4]), __uint_as_float(src[5]));
        pk.w = pack_bf16x2(__uint_as_float(src[6]), __uint_as_float(src[7]));
        *reinterpret_cast<uint4*>(op + c * 8) = pk;
      }
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc<64>(tmem);
  }
}

int launch_prefill_umma(const bf16* qkv, bf16* out, int B, int S, int H, float scale, int causal, const KvCache& c, int layer,
                        const int* block_table, int pos0, int write_cache, const uint8_t* key_mask, cudaStream_t s) {
  static bool configured_dev[kMaxDevices] = {};
  bool& configured = configured_dev[current_device_slot()];
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(attention_prefill_umma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kUmmaAttnSmem);
    if (e != cudaSuccess) return (int)e;
    configured = true;
  }
  cudaError_t e = launch_kernel(attention_prefill_umma_kernel, dim3(H, B), dim3(128), kUmmaAttnSmem, s, true, qkv, out, S, H, scale, causal,
                                c, layer, block_table, pos0, write_cache, key_mask);
  return e == cudaSuccess ? 0 : (int)e;
}

template <int NT>
int dispatch_prefill_mma_ks(int ks, const bf16* qkv, bf16* out, int B, int S, int H, int hd, float scale, int causal,
                            const KvCache& c, int layer, const int* bt, int pos0, int wc, const uint8_t* km, int rd, cudaStream_t s) {
  if (ks <= 4) return launch_prefill_mma<NT, 4>(qkv, out, B, S, H, hd, scale, causal, c, layer, bt, pos0, wc, km, rd, s);
  if (ks <= 8) return launch_prefill_mma<NT, 8>(qkv, out, B, S, H, hd, scale, causal, c, layer, bt, pos0, wc, km, rd, s);
  if (ks <= 13) return launch_prefill_mma<NT, 13>(qkv, out, B, S, H, hd, scale, causal, c, layer, bt, pos0, wc, km, rd, s);
  return launch_prefill_mma<NT, 16>(qkv, out, B, S, H, hd, scale, causal, c, layer, bt, pos0, wc, km, rd, s);
}

// ------------------------------------------------------------------------------------------------ decode
// One WARP per (row, head); 4 warps per CTA.  The step is bound by the K/V bytes it has to read, so the kernel is
// organised for memory-level parallelism: every lane owns whole tokens (t = lane, lane + 32, ...) and fetches their
// 128..512-byte K (then V) rows with independent 16-byte loads (HD/8 in flight per token slot), instead of a few
// lanes sharing one token behind a block-table lookup chain.
//   pass 1: s_t = q . K_t for the lane's tokens (q pre-scaled, fp32 in shared memory, read as broadcasts)
//   softmax statistics across the warp (+ the new token, whose k/v come from the qkv buffer, not the cache)
//   pass 2: per 64-dim chunk, acc[64] += p_t * V_t over the lane's tokens, then a 62-shuffle transpose-reduce
//           leaves dims (2*lane, 2*lane+1) of the chunk in each lane -> one coalesced 128-byte store per warp.
constexpr int kDecodeWarps = 4;

template <int HD>
__global__ void __launch_bounds__(kDecodeWarps * 32) attention_decode_kernel(
    const bf16* __restrict__ qkv, bf16* __restrict__ out, int rows, int H, float scale, KvCache cache, int layer,
    const int* __restrict__ block_table, const int* __restrict__ ctx_len, int rotary_dim, int sc_cap, long long ldo) {
  constexpr int E = HD / 32;  // dims per lane in the "own dims" layout (2, 4, 8): pairs stay inside a lane
  extern __shared__ float dsm[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  ptx::grid_dep_wait();
  ptx::grid_dep_launch();
  const int unit = blockIdx.x * kDecodeWarps + warp;  // (row, head)
  if (unit >= rows * H) return;
  const int b = unit / H, h = unit % H;
  const int d = H * HD;
  float* qs = dsm + warp * (HD + sc_cap);  // [HD] scaled query
  float* sc = qs + HD;                      // [ctx] scores
  const int ctx = ctx_len[b];               // tokens already cached; the new token sits at position ctx
  const bf16* row = qkv + static_cast<size_t>(b) * 3 * d;
  const int* bt = block_table + static_cast<size_t>(b) * cache.max_pages_per_row;

  // ---- q / k_new / v_new for this lane's E dims; rotary on q and k_new; append k_new / v_new to the cache
  float s_new = 0.f;
  {
    float q[E], kn[E], vn[E];
#pragma unroll
    for (int e = 0; e < E; e += 2) {
      const int dim = lane * E + e;
      float2 qf = unpack_bf16x2(*reinterpret_cast<const uint32_t*>(row + h * HD + dim));
      float2 kf = unpack_bf16x2(*reinterpret_cast<const uint32_t*>(row + d + h * HD + dim));
      const float2 vf = unpack_bf16x2(*reinterpret_cast<const uint32_t*>(row + 2 * d + h * HD + dim));
      if (rotary_dim > 0 && dim < rotary_dim) {
        rotary_pair(qf.x, qf.y, dim / 2, ctx, rotary_dim);
        rotary_pair(kf.x, kf.y, dim / 2, ctx, rotary_dim);
        kf = unpack_bf16x2(pack_bf16x2(kf.x, kf.y));  // exactly what later steps read back from the cache
      }
      q[e] = qf.x * scale; q[e + 1] = qf.y * scale;
      kn[e] = kf.x; kn[e + 1] = kf.y;
      vn[e] = vf.x; vn[e + 1] = vf.y;
    }
    const int page = bt[ctx / cache.page_tokens];
    const int tin = ctx % cache.page_tokens;
    bf16* kdst = cache.base + kv_index(cache, layer, 0, page, h, tin) + lane * E;
    bf16* vdst = cache.base + kv_index(cache, layer, 1, page, h, tin) + lane * E;
#pragma unroll
    for (int e = 0; e < E; e += 2) {
      *reinterpret_cast<uint32_t*>(kdst + e) = pack_bf16x2(kn[e], kn[e + 1]);
      *reinterpret_cast<uint32_t*>(vdst + e) = pack_bf16x2(vn[e], vn[e + 1]);
      qs[lane * E + e] = q[e];
      qs[lane * E + e + 1] = q[e + 1];
      s_new = fmaf(q[e], kn[e], s_new);
      s_new = fmaf(q[e + 1], kn[e + 1], s_new);
    }
    s_new = warp_sum(s_new);
  }
  __syncwarp();

  // ---- pass 1: scores of the cached tokens
  float mx = s_new;
  for (int t = lane; t < ctx; t += 32) {
    const int page = bt[t / cache.page_tokens];
    const uint4* kp = reinterpret_cast<const uint4*>(cache.base + kv_index(cache, layer, 0, page, h, t % cache.page_tokens));
    uint4 kk[HD / 8];
#pragma unroll
    for (int c = 0; c < HD / 8; ++c) kk[c] = ptx::ld_nc_u4(kp + c);
    float s = 0.f;
#pragma unroll
    for (int c = 0; c < HD / 8; ++c) {
      const float4 q0 = *reinterpret_cast<const float4*>(qs + c * 8);
      const float4 q1 = *reinterpret_cast<const float4*>(qs + c * 8 + 4);
      const float2 k0 = unpack_bf16x2(kk[c].x), k1 = unpack_bf16x2(kk[c].y), k2 = unpack_bf16x2(kk[c].z), k3 = unpack_bf16x2(kk[c].w);
      s = fmaf(q0.x, k0.x, s); s = fmaf(q0.y, k0.y, s); s = fmaf(q0.z, k1.x, s); s = fmaf(q0.w, k1.y, s);
      s = fmaf(q1.x, k2.x, s); s = fmaf(q1.y, k2.y, s); s = fmaf(q1.z, k3.x, s); s = fmaf(q1.w, k3.y, s);
    }
    sc[t] = s;
    mx = fmaxf(mx, s);
  }
  mx = warp_max(mx);
  const float p_new = expf(s_new - mx);
  float lsum = 0.f;
  for (int t = lane; t < ctx; t += 32) {
    const float p = expf(sc[t] - mx);
    sc[t] = p;  // own slots only: no cross-lane hazard
    lsum += p;
  }
  lsum = warp_sum(lsum) + p_new;
  const float inv = 1.f / lsum;

  // ---- pass 2: output, 64 dims at a time
#pragma unroll 1
  for (int c0 = 0; c0 < HD; c0 += 64) {
    float acc[64];
#pragma unroll
    for (int j = 0; j < 64; ++j) acc[j] = 0.f;
    for (int t = lane; t < ctx; t += 32) {
      const int page = bt[t / cache.page_tokens];
      const uint4* vp = reinterpret_cast<const uint4*>(cache.base + kv_index(cache, layer, 1, page, h, t % cache.page_tokens) + c0);
      uint4 vv[8];
#pragma unroll
      for (int c = 0; c < 8; ++c) vv[c] = ptx::ld_nc_u4(vp + c);
      const float p = sc[t];
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const float2 v0 = unpack_bf16x2(vv[c].x), v1 = unpack_bf16x2(vv[c].y), v2 = unpack_bf16x2(vv[c].z), v3 = unpack_bf16x2(vv[c].w);
        acc[c * 8 + 0] = fmaf(p, v0.x, acc[c * 8 + 0]); acc[c * 8 + 1] = fmaf(p, v0.y, acc[c * 8 + 1]);
        acc[c * 8 + 2] = fmaf(p, v1.x, acc[c * 8 + 2]); acc[c * 8 + 3] = fmaf(p, v1.y, acc[c * 8 + 3]);
        acc[c * 8 + 4] = fmaf(p, v2.x, acc[c * 8 + 4]); acc[c * 8 + 5] = fmaf(p, v2.y, acc[c * 8 + 5]);
        acc[c * 8 + 6] = fmaf(p, v3.x, acc[c * 8 + 6]); acc[c * 8 + 7] = fmaf(p, v3.y, acc[c * 8 + 7]);
      }
    }
    // transpose-reduce over the 32 lanes: after the round with step s a lane keeps the half of the remaining
    // dims selected by its bit s, so the survivors of lane l are dims 2l and 2l+1 of this chunk
#pragma unroll
    for (int step = 16, half = 32; step >= 1; step >>= 1, half >>= 1) {
      const bool up = (lane & step) != 0;
#pragma unroll
      for (int j = 0; j < half; ++j) {
        const float keep = up ? acc[j + half] : acc[j];
        const float send = up ? acc[j] : acc[j + half];
        acc[j] = keep + __shfl_xor_sync(0xffffffffu, send, step);
      }
    }
    const int dim = c0 + 2 * lane;
    const float2 vn = unpack_bf16x2(*reinterpret_cast<const uint32_t*>(row + 2 * d + h * HD + dim));
    const float o0 = (acc[0] + p_new * vn.x) * inv, o1 = (acc[1] + p_new * vn.y) * inv;
    *reinterpret_cast<uint32_t*>(out + static_cast<size_t>(b) * ldo + h * HD + dim) = pack_bf16x2(o0, o1);
  }
}

// ------------------------------------------------------------------------------------------------ decode, one CTA per unit
// attention_decode_kernel gives a (row, head) unit to ONE warp with lane = token: at head_dim 256 (GPT-J) a lane holds a
// whole 512-byte K row in registers and walks V in four 64-dim chunks, i.e. ~10 dependent HBM round trips per unit, on a
// grid of rows x heads / 4 CTAs (64 CTAs for 16 rows): 31 us per layer against 2 us of K/V traffic.  Here a unit gets a
// whole CTA of 128 threads and ALL its K and V rows are requested at once with cp.async (16-byte chunks, coalesced per
// row) into shared memory -- one HBM round trip per tile of `tile` tokens -- while q / k_new / v_new (rotary, cache
// append) are prepared underneath.  Scores: CH = HD / 8 lanes per token (one 16-byte chunk each), reduced by shuffles;
// softmax over the tile through shared memory; output: thread = 2 dims, walking the tile's V rows in shared memory
// (conflict-free 4-byte reads).  Tiles are folded with an online softmax; the new token is added last.
constexpr int kWideThreads = 128;

template <int HD>
__global__ void __launch_bounds__(kWideThreads) attention_decode_wide_kernel(
    const bf16* __restrict__ qkv, bf16* __restrict__ out, int rows, int H, float scale, KvCache cache, int layer,
    const int* __restrict__ block_table, const int* __restrict__ ctx_len, int rotary_dim, int tile, long long ldo) {
  constexpr int CH = HD / 8;            // 16-byte chunks per K / V row
  constexpr int TPW = 32 / CH;          // tokens a warp scores per iteration (CH <= 32)
  constexpr int NW = kWideThreads / 32;
  extern __shared__ __align__(16) uint8_t wsm[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  uint8_t* Ks = wsm;                                          // [tile][HD] bf16
  uint8_t* Vs = wsm + static_cast<size_t>(tile) * HD * 2;     // [tile][HD] bf16
  float* qs = reinterpret_cast<float*>(Vs + static_cast<size_t>(tile) * HD * 2);   // [HD]
  float* sc = qs + HD;                                        // [tile]
  float* red = sc + tile;                                     // [2 * NW]
  // Launched behind the q/k/v GEMM of the layer with programmatic stream serialization.  The context length, the block
  // table and the CACHED K / V rows do not depend on that GEMM (they were written by earlier steps; everything up to the
  // previous layer's last GEMM is complete once this kernel is resident, because the LayerNorm in between waits before it
  // lets its successor start): they are requested before the dependency wait, so the HBM round trips of the first tile
  // run underneath the GEMM's tail on every SM that has room for this CTA.  Only q / k_new / v_new wait.
  ptx::grid_dep_launch();
  const int unit = blockIdx.x;
  const int b = unit / H, h = unit - b * H;
  const int d = H * HD;
  const int ctx = ctx_len[b];
  const bf16* row = qkv + static_cast<size_t>(b) * 3 * d;
  const int* bt = block_table + static_cast<size_t>(b) * cache.max_pages_per_row;
  const uint32_t ks_u32 = ptx::smem_u32(Ks), vs_u32 = ptx::smem_u32(Vs);

  auto issue_tile = [&](int t0) {   // all K and V chunks of tokens [t0, min(ctx, t0 + tile))
    int n = ctx - t0;
    if (n > tile) n = tile;
    for (int i = tid; i < n * CH; i += kWideThreads) {
      const int j = i / CH, c = i - j * CH, t = t0 + j;
      const int page = bt[t / cache.page_tokens], tin = t % cache.page_tokens;
      const bf16* kp = cache.base + kv_index(cache, layer, 0, page, h, tin) + c * 8;
      const bf16* vp = cache.base + kv_index(cache, layer, 1, page, h, tin) + c * 8;
      const uint32_t off = static_cast<uint32_t>(j) * (HD * 2) + c * 16;
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(ks_u32 + off), "l"(kp) : "memory");
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(vs_u32 + off), "l"(vp) : "memory");
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  issue_tile(0);
  ptx::grid_dep_wait();

  // ---- q / k_new / v_new: thread owns dims (2 tid, 2 tid + 1); rotary on q and k_new; append to the cache
  float vnx = 0.f, vny = 0.f, s_part = 0.f;
  if (2 * tid < HD) {
    const int dim = 2 * tid;
    float2 qf = unpack_bf16x2(*reinterpret_cast<const uint32_t*>(row + h * HD + dim));
    float2 kf = unpack_bf16x2(*reinterpret_cast<const uint32_t*>(row + d + h * HD + dim));
    const uint32_t vw = *reinterpret_cast<const uint32_t*>(row + 2 * d + h * HD + dim);
    if (rotary_dim > 0 && dim < rotary_dim) {
      rotary_pair(qf.x, qf.y, dim / 2, ctx, rotary_dim);
      rotary_pair(kf.x, kf.y, dim / 2, ctx, rotary_dim);
      kf = unpack_bf16x2(pack_bf16x2(kf.x, kf.y));  // exactly what later steps read back from the cache
    }
    const int page = bt[ctx / cache.page_tokens], tin = ctx % cache.page_tokens;
    *reinterpret_cast<uint32_t*>(cache.base + kv_index(cache, layer, 0, page, h, tin) + dim) = pack_bf16x2(kf.x, kf.y);
    *reinterpret_cast<uint32_t*>(cache.base + kv_index(cache, layer, 1, page, h, tin) + dim) = vw;
    const float2 vf = unpack_bf16x2(vw);
    vnx = vf.x; vny = vf.y;
    qs[dim] = qf.x * scale;
    qs[dim + 1] = qf.y * scale;
    s_part = (qf.x * scale) * kf.x + (qf.y * scale) * kf.y;
  }
  s_part = warp_sum(s_part);
  if (lane == 0) red[warp] = s_part;
  __syncthreads();
  float s_new = 0.f;
#pragma unroll
  for (int w = 0; w < NW; ++w) s_new += red[w];
  // this lane's 8 query values for the score loop
  const int grp = lane / CH, ch = lane - grp * CH;
  float q8[8];
  {
    const float4 a0 = *reinterpret_cast<const float4*>(qs + ch * 8), a1 = *reinterpret_cast<const float4*>(qs + ch * 8 + 4);
    q8[0] = a0.x; q8[1] = a0.y; q8[2] = a0.z; q8[3] = a0.w; q8[4] = a1.x; q8[5] = a1.y; q8[6] = a1.z; q8[7] = a1.w;
  }

  float m_run = s_new, l_run = 0.f, accx = 0.f, accy = 0.f;
#pragma unroll 1
  for (int t0 = 0; t0 < ctx; t0 += tile) {
    int n = ctx - t0;
    if (n > tile) n = tile;
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncthreads();   // the tile has landed; (second tile on) the previous tile's red[] / sc[] reads are complete
    // ---- scores of the tile
    float mx = -INFINITY;
    for (int j0 = warp * TPW; j0 < n; j0 += NW * TPW) {
      const int j = j0 + grp;
      float sdot = 0.f;
      if (j < n) {
        const uint4 kk = *reinterpret_cast<const uint4*>(Ks + static_cast<size_t>(j) * (HD * 2) + ch * 16);
        const float2 k0 = unpack_bf16x2(kk.x), k1 = unpack_bf16x2(kk.y), k2 = unpack_bf16x2(kk.z), k3 = unpack_bf16x2(kk.w);
        sdot = q8[0] * k0.x;
        sdot = fmaf(q8[1], k0.y, sdot); sdot = fmaf(q8[2], k1.x, sdot); sdot = fmaf(q8[3], k1.y, sdot);
        sdot = fmaf(q8[4], k2.x, sdot); sdot = fmaf(q8[5], k2.y, sdot); sdot = fmaf(q8[6], k3.x, sdot); sdot = fmaf(q8[7], k3.y, sdot);
      }
#pragma unroll
      for (int o = CH / 2; o > 0; o >>= 1) sdot += __shfl_xor_sync(0xffffffffu, sdot, o);
      if (j < n) {
        if (ch == 0) sc[j] = sdot;
        mx = fmaxf(mx, sdot);
      }
    }
    mx = warp_max(mx);
    if (lane == 0) red[warp] = mx;
    __syncthreads();
    float m_new = m_run;
#pragma unroll
    for (int w = 0; w < NW; ++w) m_new = fmaxf(m_new, red[w]);
    // ---- probabilities (each thread its own slots), their sum
    float ls = 0.f;
    for (int j = tid; j < n; j += kWideThreads) {
      const float pr = expf(sc[j] - m_new);
      sc[j] = pr;
      ls += pr;
    }
    ls = warp_sum(ls);
    if (lane == 0) red[NW + warp] = ls;
    __syncthreads();
    const float resc = expf(m_run - m_new);
    float lt = 0.f;
#pragma unroll
    for (int w = 0; w < NW; ++w) lt += red[NW + w];
    l_run = l_run * resc + lt;
    m_run = m_new;
    // ---- output dims of this thread over the tile
    if (2 * tid < HD) {
      float ax = 0.f, ay = 0.f;
      const uint8_t* vcol = Vs + tid * 4;
#pragma unroll 4
      for (int j = 0; j < n; ++j) {
        const float2 vf = unpack_bf16x2(*reinterpret_cast<const uint32_t*>(vcol + static_cast<size_t>(j) * (HD * 2)));
        const float pr = sc[j];
        ax = fmaf(pr, vf.x, ax);
        ay = fmaf(pr, vf.y, ay);
      }
      accx = accx * resc + ax;
      accy = accy * resc + ay;
    }
    if (t0 + tile < ctx) {
      __syncthreads();   // every thread is done with Ks / Vs / sc before the next tile overwrites them
      issue_tile(t0 + tile);
    }
  }
  // ---- the new token (m_run >= s_new by construction)
  const float p_new = expf(s_new - m_run);
  l_run += p_new;
  if (2 * tid < HD) {
    const float inv = 1.f / l_run;
    const float o0 = (accx + p_new * vnx) * inv, o1 = (accy + p_new * vny) * inv;
    *reinterpret_cast<uint32_t*>(out + static_cast<size_t>(b) * ldo + h * HD + 2 * tid) = pack_bf16x2(o0, o1);
  }
}

// CCB_ATTN_MMA=0 sends every S <= 256 shape to the scalar kernel, CCB_ATTN_UMMA=0 the head_dim-64 S <= 64 ones to mma.sync
bool attn_use_mma() {
  static const bool on = [] {
    const char* e = getenv("CCB_ATTN_MMA");
    return !(e && e[0] == '0');
  }();
  return on;
}
bool attn_use_umma() {
  static const bool on = [] {
    const char* e = getenv("CCB_ATTN_UMMA");
    return !(e && e[0] == '0');
  }();
  return on;
}
bool attn_mma_wide(int S, int hd, int rotary_dim) {   // head_dim 264..512 on mma.sync (Q fragments streamed)
  return attn_use_mma() && S <= 80 && hd % 8 == 0 && hd > 256 && hd <= 512 && rotary_dim == 0;
}
bool attn_mma(int S, int hd, int rotary_dim) {
  return attn_use_mma() && S <= 128 && hd % 8 == 0 && hd <= 256 && rotary_dim % 2 == 0;
}
// dynamic shared memory of the scalar kernel: K (padded rows) and V of the head, per-warp q row and probability row
size_t scalar_prefill_smem(int S, int hd) {
  return (static_cast<size_t>(S) * (hd / 2 + 1) + static_cast<size_t>(S) * (hd / 2) + 1) * 4 +
         static_cast<size_t>(kPrefillWarps) * (hd + S) * 4;
}
constexpr size_t kScalarPrefillSmemCap = 200 * 1024;

}  // namespace

const char* attention_prefill_unsupported(int S, int hd, int causal, bool cache, int rotary_dim, bool key_mask) {
  if (S <= 0) return nullptr;
  if (hd <= 0 || hd % 2) return "head_dim must be positive and even";
  if (S > 256) {   // the long-sequence tcgen05 kernel: plain non-causal attention only
    if (causal || cache || rotary_dim || key_mask)
      return "above 256 tokens only non-causal attention without KV cache, rotary or key mask is supported";
    if (hd % 8 || hd > 256) return "above 256 tokens head_dim must be a multiple of 8 and at most 256";
    return nullptr;
  }
  if (attn_use_mma() && attn_use_umma() && hd == 64 && S <= 64 && rotary_dim == 0) return nullptr;
  if (attn_mma_wide(S, hd, rotary_dim) || attn_mma(S, hd, rotary_dim)) return nullptr;
  if (scalar_prefill_smem(S, hd) > kScalarPrefillSmemCap)
    return "the scalar attention kernel would need more than its 200 KB of shared memory (K and V of the whole sequence)";
  return nullptr;
}

int attention_prefill(const bf16* qkv, bf16* out, int B, int S, int H, int hd, float scale, int causal,
                      const KvCache* cache, int layer, const int* block_table, int pos0, int rotary_dim,
                      const uint8_t* key_mask, cudaStream_t s) {
  if (B <= 0 || S <= 0) return 0;
  // the shapes no kernel holds are rejected here, by the same predicate ccb_create and the LM entry points check
  if (attention_prefill_unsupported(S, hd, causal, cache != nullptr, rotary_dim, key_mask != nullptr))
    return (int)cudaErrorInvalidValue;
  if (S > 256) return attention_prefill_long(qkv, out, B, S, H, hd, scale, s);   // attention_long.cu
  if (attn_use_mma() && attn_use_umma() && hd == 64 && S <= 64 && rotary_dim == 0) {   // tcgen05 / TMEM path (ViT, GPT-2 prefill)
    KvCache c;
    if (cache) c = *cache;
    return launch_prefill_umma(qkv, out, B, S, H, scale, causal, c, layer, block_table, pos0, cache != nullptr ? 1 : 0, key_mask, s);
  }
  if (attn_mma_wide(S, hd, rotary_dim)) {
    // head_dim 512 (the 4096-wide mapper of config 5): K / V of 80 keys fill 166 KB, Q fragments are streamed
    KvCache c;
    if (cache) c = *cache;
    if (cache == nullptr)
      return launch_prefill_mma<10, 32, true>(qkv, out, B, S, H, hd, scale, causal, c, layer, block_table, pos0, 0, key_mask, rotary_dim, s);
    return launch_prefill_mma<10, 32>(qkv, out, B, S, H, hd, scale, causal, c, layer, block_table, pos0, 1, key_mask, rotary_dim, s);
  }
  if (attn_mma(S, hd, rotary_dim)) {
    KvCache c;
    if (cache) c = *cache;
    const int wc = cache != nullptr ? 1 : 0;
    const int ks = (hd + 15) / 16, nt = 2 * ((S + 15) / 16);
    if (nt > 8 && nt <= 10 && ks > 8 && ks <= 13 && cache == nullptr && rotary_dim == 0)   // the mapper: 80 keys x head_dim 200
      return launch_prefill_mma<10, 13, true>(qkv, out, B, S, H, hd, scale, causal, c, layer, block_table, pos0, 0, key_mask, 0, s);
    if (nt <= 4) return dispatch_prefill_mma_ks<4>(ks, qkv, out, B, S, H, hd, scale, causal, c, layer, block_table, pos0, wc, key_mask, rotary_dim, s);
    if (nt <= 6) return dispatch_prefill_mma_ks<6>(ks, qkv, out, B, S, H, hd, scale, causal, c, layer, block_table, pos0, wc, key_mask, rotary_dim, s);
    if (nt <= 8) return dispatch_prefill_mma_ks<8>(ks, qkv, out, B, S, H, hd, scale, causal, c, layer, block_table, pos0, wc, key_mask, rotary_dim, s);
    if (nt <= 10) return dispatch_prefill_mma_ks<10>(ks, qkv, out, B, S, H, hd, scale, causal, c, layer, block_table, pos0, wc, key_mask, rotary_dim, s);
    return dispatch_prefill_mma_ks<16>(ks, qkv, out, B, S, H, hd, scale, causal, c, layer, block_table, pos0, wc, key_mask, rotary_dim, s);
  }
  // the scalar kernel: every other shape up to 256 tokens (the predicate above checked its shared memory)
  const size_t smem = scalar_prefill_smem(S, hd);
  static size_t configured_dev[kMaxDevices] = {};
  size_t& configured = configured_dev[current_device_slot()];
  if (smem > 48 * 1024 && smem > configured) {
    cudaError_t e = cudaFuncSetAttribute(attention_prefill_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         static_cast<int>(kScalarPrefillSmemCap));
    if (e != cudaSuccess) return (int)e;
    configured = kScalarPrefillSmemCap;
  }
  KvCache c;
  if (cache) c = *cache;
  attention_prefill_kernel<<<dim3(H, B), kPrefillWarps * 32, smem, s>>>(qkv, out, S, H, hd, scale, causal, c, layer,
                                                                        block_table, pos0, rotary_dim,
                                                                        cache != nullptr ? 1 : 0, key_mask);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? 0 : (int)e;
}

int attention_decode(const bf16* qkv, bf16* out, long long ldo, int B, int H, int hd, float scale, const KvCache* cache, int layer,
                     const int* block_table, const int* ctx_len, int rotary_dim, cudaStream_t s) {
  if (B <= 0) return 0;
  if (ldo < static_cast<long long>(H) * hd || (ldo & 1)) return (int)cudaErrorInvalidValue;
  if (!cache) return (int)cudaErrorInvalidValue;
  // One CTA per (row, head) for head_dim 256 (GPT-J)
  if (hd == 256) {
    // tile = tokens staged at once: the whole context when it fits (max_pages_per_row >= max_ctx), 96 KB of K + V at most
    int tile = (cache->max_pages_per_row * cache->page_tokens + 15) & ~15;
    const int cap = (96 * 1024) / (hd * 4);
    if (tile > cap) tile = cap;
    const size_t wsmem = static_cast<size_t>(tile) * hd * 4 + (hd + tile + 2 * (kWideThreads / 32)) * sizeof(float);
    static size_t configured_dev[kMaxDevices] = {};
    size_t& configured = configured_dev[current_device_slot()];
    if (wsmem > 48 * 1024 && wsmem > configured) {
      cudaError_t e = cudaFuncSetAttribute(attention_decode_wide_kernel<256>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           112 * 1024);
      if (e != cudaSuccess) return (int)e;
      configured = 112 * 1024;
    }
    cudaError_t e = launch_kernel(attention_decode_wide_kernel<256>, dim3(B * H), dim3(kWideThreads), wsmem, s, true, qkv, out,
                                  B, H, scale, *cache, layer, block_table, ctx_len, rotary_dim, tile, ldo);
    if (e == cudaSuccess) e = cudaGetLastError();
    return e == cudaSuccess ? 0 : (int)e;
  }
  // per-warp shared memory: hd floats of q + one score per cached token
  const int sc_cap = (cache->max_pages_per_row + 3) & ~3;  // max_pages_per_row == max_ctx >= any context length
  const size_t smem = static_cast<size_t>(kDecodeWarps) * (hd + sc_cap) * sizeof(float);
  if (smem > 200 * 1024) return (int)cudaErrorInvalidValue;
  const int grid = (B * H + kDecodeWarps - 1) / kDecodeWarps;
#define CCB_LAUNCH_DECODE(HDV)                                                                                      \
  do {                                                                                                              \
    static size_t configured_dev[kMaxDevices] = {};                                                                 \
    size_t& configured = configured_dev[current_device_slot()];                                                     \
    if (smem > 48 * 1024 && smem > configured) {                                                                    \
      cudaError_t e = cudaFuncSetAttribute(attention_decode_kernel<HDV>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                           200 * 1024);                                                             \
      if (e != cudaSuccess) return (int)e;                                                                          \
      configured = 200 * 1024;                                                                                      \
    }                                                                                                               \
    cudaError_t le = launch_kernel(attention_decode_kernel<HDV>, dim3(grid), dim3(kDecodeWarps * 32), smem, s, true, \
                                   qkv, out, B, H, scale, *cache, layer, block_table, ctx_len, rotary_dim, sc_cap, ldo);   \
    if (le != cudaSuccess) return (int)le;                                                                          \
  } while (0)
  if (hd == 64)
    CCB_LAUNCH_DECODE(64);
  else if (hd == 128)
    CCB_LAUNCH_DECODE(128);
  else
    return (int)cudaErrorInvalidValue;
#undef CCB_LAUNCH_DECODE
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? 0 : (int)e;
}

}  // namespace ccb
