// Persistent bf16 GEMM for the token-heavy contractions (ViT / mapper / LM prefill: hundreds to thousands of token
// rows), normal orientation only:
//
//   out[t, f] = act(sum_k X[t, k] * W[f, k] + bias[f]) + residual[t, f]      X: [tokens, K], W: [features, K], bf16
//
// One CTA per SM walks the output tiles (128 tokens x BN features, BN a runtime multiple of 32 up to 256) of its
// static round-robin share; the fp32 accumulator is double buffered in TMEM (2 x 256 columns), so the epilogue of
// tile i (tcgen05.ld -> bias / activation / residual -> 16-byte stores) runs underneath the TMA + tcgen05.mma main
// loop of tile i + 1, and the TMA ring never drains between tiles.  With K = 1600 (25 k-blocks) the one-tile-per-CTA
// kernel of gemm_sm100.cuh spent ~37 % of its time in prologue + epilogue; here both are paid once per CTA.
//
//   warps 0, 6  TMA producers (one lane each; warp 0: X 128 x 64 tiles, warp 6: W BN x 64 tiles), ring of `stages`
//   warp 1      TMEM allocation + MMA issuer (one elected lane): 4 x tcgen05.mma 128 x BN x 16 per k-block
//   warps 2..5  epilogue, one TMEM lane quadrant each
//
// BN is picked by the host (gemm.cu) to minimise the number of waves x tile width on the machine's SM count.
#pragma once
#include "gemm_sm100.cuh"

namespace ccb {

struct PersistParams {
  int tokens, features;    // valid rows of X / W (tile rows beyond are zero-filled by TMA and masked at the store)
  int k_blocks;            // K / 64
  // epilogue: out[out_row(t) * ldo + f] = act(acc[t, f] + bias[f]) + residual[out_row(t) * ldr + f]
  void* out;               // f32 or bf16
  int out_bf16;
  long long ldo;
  const float* bias;       // per feature; may be null
  const float* residual;   // f32; may be null (may alias out)
  long long ldr;
  int act;
  // row remap: out_row(t) = (t / rg_in) * rg_out + rg_off + (t % rg_in); rg_in == 0 -> identity
  int rg_in, rg_out, rg_off;
  int bn;           // tile width in features (multiple of 32, <= 256)
  int stages;       // TMA ring depth
  int m_tiles, n_tiles;
};

constexpr int kPersistThreads = 224;
constexpr int kPersistSmemBytes = 227 * 1024;

// Fused epilogue on the 32 accumulator columns [j0, j0 + 32) of token row out_row (see gemm_apply_act for why it is kept
// small).
__device__ __forceinline__ void persist_epilogue_cols(const PersistParams& p, float (&acc)[32], bool i_ok, long long out_row,
                                                      int j0, bool vec_ok) {
  if (!i_ok) return;
  if (p.bias != nullptr) {
#pragma unroll
    for (int v = 0; v < 32; ++v) acc[v] += (j0 + v < p.features) ? __ldg(p.bias + j0 + v) : 0.f;
  }
  gemm_apply_act(acc, p.act);
  if (vec_ok && j0 + 32 <= p.features) {
    if (p.residual) {
#pragma unroll
      for (int v = 0; v < 32; v += 4) {
        const float4 r4 = *reinterpret_cast<const float4*>(p.residual + out_row * p.ldr + j0 + v);
        acc[v] += r4.x; acc[v + 1] += r4.y; acc[v + 2] += r4.z; acc[v + 3] += r4.w;
      }
    }
    // Whole 32-byte sectors per store instruction where the row allows it (256-bit st.global): a 16-byte store
    // is a PARTIAL sector write, which L2 has to merge (and, for a sector that is not resident, fill from DRAM first);
    // with thread = row every lane of a store hits a different sector, so the 16-byte form doubled the write requests
    // and cost the persistent kernels 20 % although the epilogue runs underneath the main loop.
    if (p.out_bf16) {
      __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(p.out) + out_row * p.ldo + j0;
      if ((reinterpret_cast<uintptr_t>(o) & 31) == 0) {
#pragma unroll
        for (int v = 0; v < 32; v += 16) {
          uint32_t k[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) k[e] = pack_bf16x2(acc[v + 2 * e], acc[v + 2 * e + 1]);
          ptx::st_global_256(o + v, k);
        }
      } else {
#pragma unroll
        for (int v = 0; v < 32; v += 8) {
          uint4 pk;
          pk.x = pack_bf16x2(acc[v], acc[v + 1]);
          pk.y = pack_bf16x2(acc[v + 2], acc[v + 3]);
          pk.z = pack_bf16x2(acc[v + 4], acc[v + 5]);
          pk.w = pack_bf16x2(acc[v + 6], acc[v + 7]);
          *reinterpret_cast<uint4*>(o + v) = pk;
        }
      }
    } else {
      float* o = reinterpret_cast<float*>(p.out) + out_row * p.ldo + j0;
      if ((reinterpret_cast<uintptr_t>(o) & 31) == 0) {
#pragma unroll
        for (int v = 0; v < 32; v += 8) {
          uint32_t k[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) k[e] = __float_as_uint(acc[v + e]);
          ptx::st_global_256(o + v, k);
        }
      } else {
#pragma unroll
        for (int v = 0; v < 32; v += 4)
          *reinterpret_cast<float4*>(o + v) = make_float4(acc[v], acc[v + 1], acc[v + 2], acc[v + 3]);
      }
    }
  } else {
    if (p.residual) {
      float res[32];
#pragma unroll
      for (int v = 0; v < 32; ++v) res[v] = (j0 + v < p.features) ? p.residual[out_row * p.ldr + j0 + v] : 0.f;
#pragma unroll
      for (int v = 0; v < 32; ++v) acc[v] += res[v];
    }
#pragma unroll
    for (int v = 0; v < 32; ++v) {
      const int j = j0 + v;
      if (j < p.features) {
        if (p.out_bf16)
          reinterpret_cast<__nv_bfloat16*>(p.out)[out_row * p.ldo + j] = __float2bfloat16_rn(acc[v]);
        else
          reinterpret_cast<float*>(p.out)[out_row * p.ldo + j] = acc[v];
      }
    }
  }
}

// Epilogue of one accumulator tile for one warp (thread = token row after tcgen05.ld): 32-column chunks through
// persist_epilogue_cols; the accumulator buffer is handed back to the MMA issuer (`release`) after the last TMEM read,
// before the stores of the final chunk.
// (Tried and dropped: staging the chunks through shared memory for row-contiguous 128-byte stores.  The main loop
// already saturates the SM's shared-memory port -- TMA writes 48 KB and the MMAs read 48 KB per k-block, 0.38 us at
// 128 B/clk -- so the extra ld/st.shared of the epilogue warps starve: 125 us instead of 90 us on 5120 x 6400 x 1600.)
template <class Release>
__device__ __forceinline__ void persist_epilogue_tile(const PersistParams& p, uint32_t taddr, int i, int row_b0, int lane,
                                                      Release release) {
  const int BN = p.bn;
  const bool i_ok = i < p.tokens;
  long long out_row = i;
  if (p.rg_in > 0) out_row = static_cast<long long>(i / p.rg_in) * p.rg_out + p.rg_off + (i % p.rg_in);
  const bool vec_ok = ((p.ldo & 7) == 0) && (p.residual == nullptr || (p.ldr & 3) == 0);
#pragma unroll 1
  for (int c0 = 0; c0 < BN; c0 += 32) {
    const int j0 = row_b0 + c0;
    if (j0 >= p.features) break;
    uint32_t r[32];
    ptx::tmem_ld32(taddr + c0, r);
    ptx::tmem_ld_wait();
    if (c0 + 32 >= BN || j0 + 32 >= p.features) {
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) release();
    }
    float acc[32];
#pragma unroll
    for (int v = 0; v < 32; ++v) acc[v] = __uint_as_float(r[v]);
    persist_epilogue_cols(p, acc, i_ok, out_row, j0, vec_ok);
  }
}

__global__ void __launch_bounds__(kPersistThreads, 1) gemm_persist_kernel(const __grid_constant__ CUtensorMap tma_x,
                                                                         const __grid_constant__ CUtensorMap tma_w,
                                                                         const PersistParams p) {
  extern __shared__ uint8_t smem_raw[];
  const int BN = p.bn, S = p.stages;
  const uint32_t stage_bytes = 128u * 128u + static_cast<uint32_t>(BN) * 128u;
  const uint32_t smem_base = (ptx::smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_base = smem_base + static_cast<uint32_t>(S) * stage_bytes;
  // barriers: full[S], empty[S], tmem_full[2], tmem_empty[2], then the TMEM address slot
  const uint32_t full0 = bar_base, empty0 = bar_base + 8u * S;
  const uint32_t tfull0 = bar_base + 16u * S, tempty0 = tfull0 + 16u;
  const uint32_t tmem_slot = tempty0 + 16u;
  uint8_t* smem_gen = smem_raw + (smem_base - ptx::smem_u32(smem_raw));
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_gen + (tmem_slot - smem_base));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    ptx::prefetch_tmap(&tma_x);
    ptx::prefetch_tmap(&tma_w);
    for (int s = 0; s < S; ++s) {
      ptx::mbar_init(full0 + 8u * s, 1);
      ptx::mbar_init(empty0 + 8u * s, 1);
    }
    for (int b = 0; b < 2; ++b) {
      ptx::mbar_init(tfull0 + 8u * b, 1);
      ptx::mbar_init(tempty0 + 8u * b, 4);
    }
    ptx::fence_mbar_init();
  }
  if (warp == 1) ptx::tmem_alloc<512>(tmem_slot);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;
  ptx::grid_dep_launch();

  const int ntiles = p.m_tiles * p.n_tiles;
  const int nkb = p.k_blocks;

  if (warp == 0 || warp == 6) {
    // ------------------------------------------------------------ TMA producers: warp 0 loads X, warp 6 loads W
    // (one thread issues a tensor load every ~130 ns; two loads per k-block from one thread would pace the ring at
    //  the speed of the MMAs themselves, so each operand has its own issuing thread)
    {
      const bool is_x = warp == 0;
      // weights never depend on the preceding kernel: with PDL their tiles are requested ahead of the dependency wait
      if (is_x) ptx::grid_dep_wait();
      const CUtensorMap* tm = is_x ? &tma_x : &tma_w;
      const uint32_t off = is_x ? 0u : 128u * 128u;
      const uint64_t hint = is_x ? ptx::kEvictLast : ptx::kEvictNormal;
      uint32_t s = 0, ph = 0;
#pragma unroll 1
      for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int row = is_x ? (tile % p.m_tiles) * 128 : (tile / p.m_tiles) * BN;
#pragma unroll 1
        for (int kb = 0; kb < nkb; ++kb) {
          ptx::mbar_wait(empty0 + 8u * s, ph ^ 1);
          if (ptx::elect_one()) {
            if (is_x) ptx::mbar_arrive_expect_tx(full0 + 8u * s, stage_bytes);
            ptx::tma_load_2d(smem_base + s * stage_bytes + off, tm, full0 + 8u * s, kb * 64, row, hint);
          }
          __syncwarp();
          if (++s == static_cast<uint32_t>(S)) { s = 0; ph ^= 1; }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer
    // The whole (converged) warp runs the loops and waits; one elected lane issues.  Everything the issue needs is
    // warp-uniform, so the compiler keeps it in uniform registers and emits the tcgen05 instructions back to back; under
    // `if (lane == 0)` every descriptor went through R2UR and every instruction through its own election loop, which
    // cost ~0.3 us per k-block -- as much as the MMAs of a 256-wide tile and 3x those of a 64-wide one.
    {
      const uint32_t idesc = ptx::umma_idesc_bf16(128, BN);
      const uint64_t desc0 = ptx::umma_desc_k_sw128(smem_base);
      uint32_t s = 0, ph = 0, it = 0;
#pragma unroll 1
      for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
        const uint32_t buf = it & 1, aph = (it >> 1) & 1;
        ptx::mbar_wait(tempty0 + 8u * buf, aph ^ 1);   // the epilogue drained this accumulator
        ptx::tc_fence_after();
        const uint32_t tacc = tmem_base + buf * 256u;
#pragma unroll 1
        for (int kb = 0; kb < nkb; ++kb) {
          ptx::mbar_wait(full0 + 8u * s, ph);
          ptx::tc_fence_after();
          if (ptx::elect_one()) {
            const uint64_t adesc = desc0 + static_cast<uint64_t>((s * stage_bytes) >> 4);
            const uint64_t bdesc = adesc + static_cast<uint64_t>((128u * 128u) >> 4);
            ptx::umma_bf16(tacc, adesc, bdesc, idesc, kb > 0 ? 1u : 0u);
            ptx::umma_bf16(tacc, adesc + 2u, bdesc + 2u, idesc, 1u);
            ptx::umma_bf16(tacc, adesc + 4u, bdesc + 4u, idesc, 1u);
            ptx::umma_bf16(tacc, adesc + 6u, bdesc + 6u, idesc, 1u);
            ptx::umma_commit(empty0 + 8u * s);
            if (kb == nkb - 1) ptx::umma_commit(tfull0 + 8u * buf);
          }
          __syncwarp();
          if (++s == static_cast<uint32_t>(S)) { s = 0; ph ^= 1; }
        }
      }
    }
  } else {
    // ------------------------------------------------------------ epilogue warps
    ptx::grid_dep_wait();   // residual / out belong to the preceding kernels of the chain
    const int quad = warp & 3;
    uint32_t it = 0;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
      const int m_blk = tile % p.m_tiles, n_blk = tile / p.m_tiles;
      const uint32_t buf = it & 1, aph = (it >> 1) & 1;
      const int i = m_blk * 128 + quad * 32 + lane;
      ptx::mbar_wait(tfull0 + 8u * buf, aph);
      ptx::tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + buf * 256u;
      const uint32_t rel = tempty0 + 8u * buf;
      persist_epilogue_tile(p, taddr, i, n_blk * BN, lane, [rel]() { ptx::mbar_arrive(rel); });
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc<512>(tmem_base);
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// CTA-pair variant (cta_group::2): the two CTAs of a cluster (one TPC) compute one 256-token x BN-feature tile per
// tcgen05.mma.  Each CTA stages its own 128 token rows of X and HALF of the W rows of the tile, so the operand bytes an
// SM pulls from L2 per k-block drop from 16 KB + BN x 128 B to 16 KB + BN x 64 B: at 148 SMs the single-CTA kernel's
// 48 KB per 128 x 256 x 64 k-block (~14 KB/clk chip-wide at tensor peak) is more than L2 can deliver, which is what
// capped it at ~1.1 PFLOP/s.  The leader (cluster rank 0) issues the MMAs and owns the `full` and `tmem_empty`
// barriers; `empty` and `tmem_full` are signalled in both CTAs by multicast commits.
__global__ void __launch_bounds__(kPersistThreads, 1) gemm_pair_kernel(const __grid_constant__ CUtensorMap tma_x,
                                                                      const __grid_constant__ CUtensorMap tma_w,
                                                                      const PersistParams p) {
  extern __shared__ uint8_t smem_raw[];
  const int BN = p.bn, S = p.stages;
  const uint32_t w_bytes = static_cast<uint32_t>(BN) * 64u;            // BN / 2 rows x 128 B
  const uint32_t stage_bytes = 128u * 128u + w_bytes;
  const uint32_t smem_base = (ptx::smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_base = smem_base + static_cast<uint32_t>(S) * stage_bytes;
  const uint32_t full0 = bar_base, empty0 = bar_base + 8u * S;
  const uint32_t tfull0 = bar_base + 16u * S, tempty0 = tfull0 + 16u;
  const uint32_t tmem_slot = tempty0 + 16u;
  uint8_t* smem_gen = smem_raw + (smem_base - ptx::smem_u32(smem_raw));
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_gen + (tmem_slot - smem_base));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = ptx::cluster_ctarank();
  const bool leader = rank == 0;
  if (threadIdx.x == 0) {
    ptx::prefetch_tmap(&tma_x);
    ptx::prefetch_tmap(&tma_w);
    for (int s = 0; s < S; ++s) {
      ptx::mbar_init(full0 + 8u * s, 1);     // (leader's is used) the leader's expect_tx covers both CTAs' bytes
      ptx::mbar_init(empty0 + 8u * s, 1);
    }
    for (int b = 0; b < 2; ++b) {
      ptx::mbar_init(tfull0 + 8u * b, 1);
      ptx::mbar_init(tempty0 + 8u * b, 8);   // (leader's is used) 4 epilogue warps of each CTA
    }
    ptx::fence_mbar_init();
  }
  if (warp == 1) ptx::tmem_alloc_pair<512>(tmem_slot);
  ptx::tc_fence_before();
  ptx::cluster_arrive();    // barriers of both CTAs are initialised before anyone signals them
  ptx::cluster_wait();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;
  ptx::grid_dep_launch();

  const int ntiles = p.m_tiles * p.n_tiles;       // m_tiles counts 256-row pair tiles
  const int nkb = p.k_blocks;
  const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;

  if (warp == 0 || warp == 6) {
    // ------------------------------------------------------------ TMA producers (both CTAs): warp 0 loads X, warp 6 W
    {
      const bool is_x = warp == 0;
      if (is_x) ptx::grid_dep_wait();
      const CUtensorMap* tm = is_x ? &tma_x : &tma_w;
      const uint32_t off = is_x ? 0u : 128u * 128u;
      const uint64_t hint = is_x ? ptx::kEvictLast : ptx::kEvictNormal;
      const uint32_t lfull0 = ptx::mapa_shared(full0, 0);   // the leader's `full` barriers
      uint32_t s = 0, ph = 0;
#pragma unroll 1
      for (int tile = pair; tile < ntiles; tile += npairs) {
        const int row = is_x ? (tile % p.m_tiles) * 256 + static_cast<int>(rank) * 128
                             : (tile / p.m_tiles) * BN + static_cast<int>(rank) * (BN >> 1);
#pragma unroll 1
        for (int kb = 0; kb < nkb; ++kb) {
          ptx::mbar_wait(empty0 + 8u * s, ph ^ 1);
          if (ptx::elect_one()) {
            if (is_x && leader) ptx::mbar_arrive_expect_tx(full0 + 8u * s, 2u * stage_bytes);
            ptx::tma_load_2d_pair(smem_base + s * stage_bytes + off, tm, lfull0 + 8u * s, kb * 64, row, hint);
          }
          __syncwarp();
          if (++s == static_cast<uint32_t>(S)) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer (leader only; converged warp, elected issue)
    if (leader) {
      const uint32_t idesc = ptx::umma_idesc_bf16(256, BN);
      const uint64_t desc0 = ptx::umma_desc_k_sw128(smem_base);
      uint32_t s = 0, ph = 0, it = 0;
#pragma unroll 1
      for (int tile = pair; tile < ntiles; tile += npairs, ++it) {
        const uint32_t buf = it & 1, aph = (it >> 1) & 1;
        ptx::mbar_wait(tempty0 + 8u * buf, aph ^ 1);
        ptx::tc_fence_after();
        const uint32_t tacc = tmem_base + buf * 256u;
#pragma unroll 1
        for (int kb = 0; kb < nkb; ++kb) {
          ptx::mbar_wait(full0 + 8u * s, ph);
          ptx::tc_fence_after();
          if (ptx::elect_one()) {
            const uint64_t adesc = desc0 + static_cast<uint64_t>((s * stage_bytes) >> 4);
            const uint64_t bdesc = adesc + static_cast<uint64_t>((128u * 128u) >> 4);
            ptx::umma_bf16_pair(tacc, adesc, bdesc, idesc, kb > 0 ? 1u : 0u);
            ptx::umma_bf16_pair(tacc, adesc + 2u, bdesc + 2u, idesc, 1u);
            ptx::umma_bf16_pair(tacc, adesc + 4u, bdesc + 4u, idesc, 1u);
            ptx::umma_bf16_pair(tacc, adesc + 6u, bdesc + 6u, idesc, 1u);
            ptx::umma_commit_pair(empty0 + 8u * s, 3);
            if (kb == nkb - 1) ptx::umma_commit_pair(tfull0 + 8u * buf, 3);
          }
          __syncwarp();
          if (++s == static_cast<uint32_t>(S)) { s = 0; ph ^= 1; }
        }
      }
    }
  } else {
    // ------------------------------------------------------------ epilogue warps (both CTAs, own 128 token rows)
    ptx::grid_dep_wait();
    const int quad = warp & 3;
    const uint32_t ltempty0 = ptx::mapa_shared(tempty0, 0);
    uint32_t it = 0;
    for (int tile = pair; tile < ntiles; tile += npairs, ++it) {
      const int m_blk = tile % p.m_tiles, n_blk = tile / p.m_tiles;
      const uint32_t buf = it & 1, aph = (it >> 1) & 1;
      const int i = m_blk * 256 + static_cast<int>(rank) * 128 + quad * 32 + lane;
      ptx::mbar_wait(tfull0 + 8u * buf, aph);
      ptx::tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + buf * 256u;
      const uint32_t rel = ltempty0 + 8u * buf;
      persist_epilogue_tile(p, taddr, i, n_blk * BN, lane, [rel]() { ptx::mbar_arrive_cluster(rel); });
    }
  }

  ptx::tc_fence_before();
  ptx::cluster_arrive();    // the peer may still be signalling the leader's barriers / reading its accumulator
  ptx::cluster_wait();
  if (warp == 1) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc_pair<512>(tmem_base);
  }
}

}  // namespace ccb
