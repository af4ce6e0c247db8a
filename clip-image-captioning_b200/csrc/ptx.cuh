// Thin inline-PTX wrappers for sm_100a: mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (alloc / mma /
// commit / ld) and a few cache-hinted global accesses.  Everything here is device-only plumbing used by
// the GEMM and streaming kernels of libclipcap_b200.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace ccb {
namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ uint64_t globaltimer_ns() {
  uint64_t t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ uint32_t mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t done;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(done)
      : "r"(bar), "r"(parity)
      : "memory");
  return done;
}
// Bounded wait: a protocol bug traps (launch fails with an error) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const uint64_t t0 = globaltimer_ns();
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if ((++spins & 0x3ff) == 0 && globaltimer_ns() - t0 > 4000000000ull) __trap();
  }
}

// ---------------------------------------------------------------- TMA
constexpr uint64_t kEvictFirst = 0x12F0000000000000ull;
constexpr uint64_t kEvictNormal = 0x1000000000000000ull;
constexpr uint64_t kEvictLast = 0x14F0000000000000ull;

__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t smem_dst, const CUtensorMap* m, uint32_t bar, int c0, int c1,
                                            uint64_t hint) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4}], [%2], %5;"
      ::"r"(smem_dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1), "l"(hint)
      : "memory");
}

// ---------------------------------------------------------------- tcgen05 / TMEM
template <int kCols>
__device__ __forceinline__ void tmem_alloc(uint32_t smem_slot) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_slot), "n"(kCols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int kCols>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem]^T, bf16 inputs, fp32 accumulate, issued by ONE thread.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrives (count 1) on the mbarrier once all previously issued tcgen05.mma of this thread completed.
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// 32 lanes x 32 consecutive fp32 columns: thread t of the warp receives lane (base_lane + t).
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32"
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15,"
      " %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
// 32 lanes x 8 consecutive fp32 columns
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
               : "memory");
}
// 32 lanes x 16 consecutive fp32 columns
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32"
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32"
      " [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
        "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// UMMA shared-memory descriptor for a K-major bf16 tile stored as 128-byte rows with the 128B swizzle
// (exactly what a TMA box of {64 elements, rows} with CU_TENSOR_MAP_SWIZZLE_128B writes):
//   start address>>4 | LBO (ignored for swizzled K-major) | SBO = 1024 B between 8-row groups |
//   version=1 (sm_100) | layout_type=2 (SWIZZLE_128B).
__device__ __forceinline__ uint64_t umma_desc_k_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFF) >> 4);
  d |= static_cast<uint64_t>(1) << 16;            // leading byte offset (unused) = 16 B
  d |= static_cast<uint64_t>(1024 >> 4) << 32;    // stride byte offset
  d |= static_cast<uint64_t>(1) << 46;            // descriptor version (Blackwell)
  d |= static_cast<uint64_t>(2) << 61;            // SWIZZLE_128B
  return d;
}
// The same tile read as an MN-major operand (e.g. V [keys][dims] as the B operand of P.V, N = dims, K = keys): 128-byte rows
// along K, 8-row groups SBO = 1024 B apart, successive 64-element blocks along N `lbo` bytes apart.
__device__ __forceinline__ uint64_t umma_desc_mn_sw128(uint32_t smem_addr, uint32_t lbo) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFF) >> 4);
  d |= static_cast<uint64_t>((lbo >> 4) & 0x3FFF) << 16;
  d |= static_cast<uint64_t>(1024 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}
// Instruction descriptor, kind::f16: D=f32, A=B=bf16, both K-major, shape M x N (K fixed at 16).
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N) {
  return (1u << 4)                       // c_format  = F32
         | (1u << 7)                     // a_format  = BF16
         | (1u << 10)                    // b_format  = BF16
         | (0u << 15) | (0u << 16)       // a_major = b_major = K
         | (static_cast<uint32_t>(N >> 3) << 17) | (static_cast<uint32_t>(M >> 4) << 24);
}


// ---------------------------------------------------------------- CTA pairs (cta_group::2)
// Two CTAs of one cluster (ranks 0 / 1, one TPC) issue ONE tcgen05.mma of M = 256: each CTA holds its 128 rows of A,
// its half of the B rows and its 128 accumulator lanes; the instruction is issued by the leader (rank 0) only, with
// shared-memory descriptors relative to the leader's window (the peer uses the same offsets).
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
template <int kCols>
__device__ __forceinline__ void tmem_alloc_pair(uint32_t smem_slot) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_slot), "n"(kCols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <int kCols>
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols) : "memory");
}
__device__ __forceinline__ void umma_bf16_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrives on the mbarrier at this shared-memory offset in every CTA of `cta_mask` once the issued MMAs completed
__device__ __forceinline__ void umma_commit_pair(uint32_t bar, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(bar), "h"(cta_mask)
               : "memory");
}
// TMA load into THIS CTA's shared memory that completes its bytes on an mbarrier of the pair's leader
// (`bar_cluster` is a shared::cluster address, e.g. from mapa_shared(bar, 0))
__device__ __forceinline__ void tma_load_2d_pair(uint32_t smem_dst, const CUtensorMap* m, uint32_t bar_cluster, int c0, int c1,
                                                 uint64_t hint) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4}], [%2], %5;"
      ::"r"(smem_dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster), "r"(c0), "r"(c1), "l"(hint)
      : "memory");
}
// arrive (count 1) on an mbarrier given by its shared::cluster address (possibly in the peer CTA)
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t bar_cluster) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(bar_cluster) : "memory");
}

// ---------------------------------------------------------------- misc global memory
__device__ __forceinline__ float ldcg_f32(const float* p) {
  float v;
  asm volatile("ld.global.cg.f32 %0, [%1];" : "=f"(v) : "l"(p));
  return v;
}
// 256-bit store (sm_100+): one whole 32-byte sector per lane
__device__ __forceinline__ void st_global_256(void* p, const uint32_t (&v)[8]) {
  asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]),
               "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
               : "memory");
}
__device__ __forceinline__ uint4 ld_nc_u4(const void* p) {
  uint4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
               : "l"(p));
  return v;
}

// ---------------------------------------------------------------- programmatic dependent launch
// wait: blocks until the kernel this one was launched behind (with programmatic stream serialization) has fully
// completed and its memory is visible; a no-op for a normal launch.  launch_dependents: lets the NEXT kernel of
// the stream start its prologue (everything before its own wait) while this one is still running.
__device__ __forceinline__ void grid_dep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void grid_dep_launch() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// ---------------------------------------------------------------- clusters / distributed shared memory
__device__ __forceinline__ void cluster_arrive() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }
// shared::cta address of this CTA -> shared::cluster address of the same offset in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_shared(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ float ld_dsmem_f32(uint32_t addr) {
  float v;
  asm volatile("ld.shared::cluster.f32 %0, [%1];" : "=f"(v) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ void st_dsmem_f32(uint32_t addr, float v) {
  asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory");
}
__device__ __forceinline__ float ld_shared_f32(uint32_t addr) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ void st_shared_f32(uint32_t addr, float v) {
  asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory");
}

// one lane of the (converged) warp: the way single-thread instructions (TMA, tcgen05.mma / commit) are issued
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

}  // namespace ptx
}  // namespace ccb
