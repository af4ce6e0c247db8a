// Row-wise and glue kernels: LayerNorm, ViT patchify / token assembly, mapper constant rows, embedding
// gathers.  All are HBM/L2-bound streaming kernels: 16-byte vector accesses, one CTA per row.
#include <stdlib.h>

#include "common.cuh"
#include "internal.h"
#include "ptx.cuh"

namespace ccb {

namespace {

#define CCB_LAUNCH_CHECK()                         \
  do {                                             \
    cudaError_t e__ = cudaGetLastError();          \
    if (e__ != cudaSuccess) return (int)e__;       \
  } while (0)

// ---------------------------------------------------------------- LayerNorm
// One CTA per row; the row is staged in shared memory (d * 4 bytes) so x is read from HBM exactly once.
template <typename OutT>
__global__ void __launch_bounds__(256) layernorm_kernel(const float* __restrict__ x, long long ldx,
                                                        const float* __restrict__ gamma,
                                                        const float* __restrict__ beta, float eps,
                                                        OutT* __restrict__ y, long long ldy, int d) {
  extern __shared__ float row[];
  __shared__ float scratch[32];
  ptx::grid_dep_wait();
  ptx::grid_dep_launch();
  const float* xr = x + static_cast<long long>(blockIdx.x) * ldx;
  if (d <= 4 * 4 * static_cast<int>(blockDim.x) && blockDim.x == 256) {
    // up to four 16-byte chunks per thread (d <= 4096): the row, gamma and beta are all requested before anything is
    // used -- ONE L2 round trip where the loops below have one per iteration (eight at d = 4096: this kernel is on the
    // critical path of every layer of the operator-chain decode step).  Same summation order as the loops.
    float4 v[4], g[4], bb[4];
    const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int c = (threadIdx.x + i * 256) * 4;
      const bool ok = c < d;
      v[i] = ok ? *reinterpret_cast<const float4*>(xr + c) : z4;
      g[i] = ok ? __ldg(reinterpret_cast<const float4*>(gamma + c)) : z4;
      bb[i] = ok ? __ldg(reinterpret_cast<const float4*>(beta + c)) : z4;
    }
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 4; ++i)
      if ((threadIdx.x + i * 256) * 4 < d) s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
    const float mean = block_sum(s, scratch) / d;
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      if ((threadIdx.x + i * 256) * 4 < d) {
        const float a = v[i].x - mean, b = v[i].y - mean, cc = v[i].z - mean, dd = v[i].w - mean;
        q += (a * a + b * b) + (cc * cc + dd * dd);
      }
    }
    const float var = block_sum(q, scratch) / d;
    const float rstd = rsqrtf(var + eps);
    OutT* yr = y + static_cast<long long>(blockIdx.x) * ldy;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int c = (threadIdx.x + i * 256) * 4;
      if (c < d) {
        const float o0 = (v[i].x - mean) * rstd * g[i].x + bb[i].x;
        const float o1 = (v[i].y - mean) * rstd * g[i].y + bb[i].y;
        const float o2 = (v[i].z - mean) * rstd * g[i].z + bb[i].z;
        const float o3 = (v[i].w - mean) * rstd * g[i].w + bb[i].w;
        if constexpr (sizeof(OutT) == 2) {
          uint2 pk;
          pk.x = pack_bf16x2(o0, o1);
          pk.y = pack_bf16x2(o2, o3);
          *reinterpret_cast<uint2*>(yr + c) = pk;
        } else {
          *reinterpret_cast<float4*>(yr + c) = make_float4(o0, o1, o2, o3);
        }
      }
    }
    return;
  }
  float s = 0.f;
  for (int c = threadIdx.x * 4; c < d; c += blockDim.x * 4) {
    const float4 v = *reinterpret_cast<const float4*>(xr + c);
    *reinterpret_cast<float4*>(row + c) = v;
    s += (v.x + v.y) + (v.z + v.w);
  }
  const float mean = block_sum(s, scratch) / d;
  float q = 0.f;
  for (int c = threadIdx.x * 4; c < d; c += blockDim.x * 4) {
    const float4 v = *reinterpret_cast<const float4*>(row + c);
    const float a = v.x - mean, b = v.y - mean, cc = v.z - mean, dd = v.w - mean;
    q += (a * a + b * b) + (cc * cc + dd * dd);
  }
  const float var = block_sum(q, scratch) / d;
  const float rstd = rsqrtf(var + eps);
  OutT* yr = y + static_cast<long long>(blockIdx.x) * ldy;
  for (int c = threadIdx.x * 4; c < d; c += blockDim.x * 4) {
    const float4 v = *reinterpret_cast<const float4*>(row + c);
    const float4 g = __ldg(reinterpret_cast<const float4*>(gamma + c));
    const float4 b = __ldg(reinterpret_cast<const float4*>(beta + c));
    const float o0 = (v.x - mean) * rstd * g.x + b.x;
    const float o1 = (v.y - mean) * rstd * g.y + b.y;
    const float o2 = (v.z - mean) * rstd * g.z + b.z;
    const float o3 = (v.w - mean) * rstd * g.w + b.w;
    if constexpr (sizeof(OutT) == 2) {
      uint2 pk;
      pk.x = pack_bf16x2(o0, o1);
      pk.y = pack_bf16x2(o2, o3);
      *reinterpret_cast<uint2*>(yr + c) = pk;
    } else {
      *reinterpret_cast<float4*>(yr + c) = make_float4(o0, o1, o2, o3);
    }
  }
}

// One WARP per row, the row held in registers (NV float4 per lane): no shared memory, no block barrier, all loads of
// a row in flight at once.  With thousands of rows (ViT / mapper / prefill) the one-CTA-per-row kernel above is a chain
// of two block reductions per CTA and runs in waves; here every row of the call is resident at once.
template <int NV>
__global__ void __launch_bounds__(256) layernorm_rows_kernel(const float* __restrict__ x, long long ldx,
                                                             const float* __restrict__ gamma, const float* __restrict__ beta,
                                                             float eps, bf16* __restrict__ y, long long ldy, int rows, int d) {
  ptx::grid_dep_wait();
  ptx::grid_dep_launch();
  const int lane = threadIdx.x & 31;
  const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= rows) return;
  const int nq = d >> 2;
  const float4* xr = reinterpret_cast<const float4*>(x + static_cast<long long>(r) * ldx);
  float4 v[NV];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int q = lane + 32 * i;
    v[i] = q < nq ? xr[q] : make_float4(0.f, 0.f, 0.f, 0.f);
    s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
  }
  const float mean = warp_sum(s) / d;
  float qs = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    if (lane + 32 * i < nq) {
      const float a = v[i].x - mean, b = v[i].y - mean, c = v[i].z - mean, e = v[i].w - mean;
      qs += (a * a + b * b) + (c * c + e * e);
    }
  }
  const float rstd = rsqrtf(warp_sum(qs) / d + eps);
  uint2* yr = reinterpret_cast<uint2*>(y + static_cast<long long>(r) * ldy);
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int q = lane + 32 * i;
    if (q < nq) {
      const float4 g = __ldg(reinterpret_cast<const float4*>(gamma) + q);
      const float4 b = __ldg(reinterpret_cast<const float4*>(beta) + q);
      uint2 pk;
      pk.x = pack_bf16x2((v[i].x - mean) * rstd * g.x + b.x, (v[i].y - mean) * rstd * g.y + b.y);
      pk.y = pack_bf16x2((v[i].z - mean) * rstd * g.z + b.z, (v[i].w - mean) * rstd * g.w + b.w);
      yr[q] = pk;
    }
  }
}

// ---------------------------------------------------------------- ViT patchify (im2col for stride == kernel)
template <typename InT>
__device__ __forceinline__ float to_f32(InT v);
template <>
__device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <>
__device__ __forceinline__ float to_f32<__half>(__half v) { return __half2float(v); }
template <>
__device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }

template <typename InT>
__global__ void __launch_bounds__(256) patchify_kernel(const InT* __restrict__ img, int B, int C, int H, int W,
                                                       int ps, bf16* __restrict__ patches) {
  const int gw = W / ps, gh = H / ps;
  const int kdim = C * ps * ps;
  const long long total8 = static_cast<long long>(B) * gh * gw * kdim / 8;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total8;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long e = idx * 8;
    const int col = static_cast<int>(e % kdim);
    const long long prow = e / kdim;
    const int px = static_cast<int>(prow % gw);
    const int py = static_cast<int>((prow / gw) % gh);
    const int b = static_cast<int>(prow / (gw * gh));
    const int kx = col % ps, ky = (col / ps) % ps, c = col / (ps * ps);
    const InT* src = img + ((static_cast<long long>(b) * C + c) * H + (py * ps + ky)) * W + px * ps + kx;
    float v[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) v[q] = to_f32<InT>(src[q]);
    uint4 pk;
    pk.x = pack_bf16x2(v[0], v[1]);
    pk.y = pack_bf16x2(v[2], v[3]);
    pk.z = pack_bf16x2(v[4], v[5]);
    pk.w = pack_bf16x2(v[6], v[7]);
    *reinterpret_cast<uint4*>(patches + e) = pk;
  }
}

// Patch sizes whose row is not a multiple of 8 pixels (ViT-L/14: 14): one element per thread, rows written at pitch
// ldp >= kdim (the GEMM's K, a multiple of 64) with zeros in the pad columns.
template <typename InT>
__global__ void __launch_bounds__(256) patchify_any_kernel(const InT* __restrict__ img, int B, int C, int H, int W, int ps,
                                                           int ldp, bf16* __restrict__ patches) {
  const int gw = W / ps, gh = H / ps;
  const int kdim = C * ps * ps;
  const long long total = static_cast<long long>(B) * gh * gw * ldp;
  for (long long e = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; e < total;
       e += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int col = static_cast<int>(e % ldp);
    const long long prow = e / ldp;
    float v = 0.f;
    if (col < kdim) {
      const int px = static_cast<int>(prow % gw);
      const int py = static_cast<int>((prow / gw) % gh);
      const int b = static_cast<int>(prow / (gw * gh));
      const int kx = col % ps, ky = (col / ps) % ps, c = col / (ps * ps);
      v = to_f32<InT>(img[((static_cast<long long>(b) * C + c) * H + (py * ps + ky)) * W + px * ps + kx]);
    }
    patches[e] = __float2bfloat16_rn(v);
  }
}


// ---------------------------------------------------------------- weight ingestion (cast / transpose)
template <typename InT>
__global__ void __launch_bounds__(256) convert_rows_bf16_kernel(const InT* __restrict__ src, long long rows, int cols,
                                                                bf16* __restrict__ dst, long long dst_ld) {
  const long long total = rows * cols;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long r = i / cols;
    const int c = static_cast<int>(i % cols);
    dst[r * dst_ld + c] = __float2bfloat16_rn(to_f32<InT>(src[i]));
  }
}
template <typename InT>
__global__ void __launch_bounds__(256) convert_f32_kernel(const InT* __restrict__ src, long long n,
                                                          float* __restrict__ dst) {
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x)
    dst[i] = to_f32<InT>(src[i]);
}
// src [R, C] -> dst [C, R] (row pitch dst_ld), through a padded 32x32 shared tile
template <typename InT>
__global__ void __launch_bounds__(256) transpose_bf16_kernel(const InT* __restrict__ src, int R, int C,
                                                             bf16* __restrict__ dst, long long dst_ld) {
  __shared__ float tile[32][33];
  const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
  for (int k = ty; k < 32; k += 8) {
    const int r = r0 + k, c = c0 + tx;
    tile[k][tx] = (r < R && c < C) ? to_f32<InT>(src[static_cast<long long>(r) * C + c]) : 0.f;
  }
  __syncthreads();
  for (int k = ty; k < 32; k += 8) {
    const int c = c0 + k, r = r0 + tx;
    if (c < C && r < R) dst[static_cast<long long>(c) * dst_ld + r] = __float2bfloat16_rn(tile[tx][k]);
  }
}

// ---------------------------------------------------------------- ViT token assembly + ln_pre
__global__ void __launch_bounds__(256) vit_assemble_kernel(const float* __restrict__ patch_emb,
                                                           const float* __restrict__ cls,
                                                           const float* __restrict__ pos,
                                                           const float* __restrict__ g, const float* __restrict__ bta,
                                                           float eps, float* __restrict__ x, int np, int d) {
  extern __shared__ float row[];
  __shared__ float scratch[32];
  const int t = blockIdx.x % (np + 1);
  const int b = blockIdx.x / (np + 1);
  const float* src = (t == 0) ? cls : patch_emb + (static_cast<long long>(b) * np + (t - 1)) * d;
  const float* pr = pos + static_cast<long long>(t) * d;
  float s = 0.f;
  for (int c = threadIdx.x; c < d; c += blockDim.x) {
    const float v = src[c] + pr[c];
    row[c] = v;
    s += v;
  }
  const float mean = block_sum(s, scratch) / d;
  float q = 0.f;
  for (int c = threadIdx.x; c < d; c += blockDim.x) {
    const float a = row[c] - mean;
    q += a * a;
  }
  const float rstd = rsqrtf(block_sum(q, scratch) / d + eps);
  float* xr = x + static_cast<long long>(blockIdx.x) * d;
  for (int c = threadIdx.x; c < d; c += blockDim.x) xr[c] = (row[c] - mean) * rstd * g[c] + bta[c];
}

__global__ void __launch_bounds__(256) mapper_fill_const_kernel(const float* __restrict__ pc, float* __restrict__ seq,
                                                                int clip_len, int P, int d) {
  // grid: (P, B)
  const int p = blockIdx.x, b = blockIdx.y;
  const float4* src = reinterpret_cast<const float4*>(pc + static_cast<long long>(p) * d);
  float4* dst = reinterpret_cast<float4*>(seq + (static_cast<long long>(b) * (clip_len + P) + clip_len + p) * d);
  for (int c = threadIdx.x; c < d / 4; c += blockDim.x) dst[c] = __ldg(src + c);
}

__global__ void __launch_bounds__(256) mapper_fill_pos_kernel(const float* __restrict__ pos, float* __restrict__ seq,
                                                              int clip_len, int P, int d) {
  // grid: (clip_len, B)
  const int t = blockIdx.x, b = blockIdx.y;
  float4* dst = reinterpret_cast<float4*>(seq + (static_cast<long long>(b) * (clip_len + P) + t) * d);
  const float4* src = pos ? reinterpret_cast<const float4*>(pos + static_cast<long long>(t) * d) : nullptr;
  for (int c = threadIdx.x; c < d / 4; c += blockDim.x) dst[c] = src ? __ldg(src + c) : make_float4(0.f, 0.f, 0.f, 0.f);
}

__global__ void __launch_bounds__(256) cast_kernel(const float* __restrict__ x, long long ldx, bf16* __restrict__ y,
                                                   long long ldy, int d) {
  const float* xr = x + static_cast<long long>(blockIdx.x) * ldx;
  bf16* yr = y + static_cast<long long>(blockIdx.x) * ldy;
  for (int c = threadIdx.x * 4; c < d; c += blockDim.x * 4) {
    const float4 v = *reinterpret_cast<const float4*>(xr + c);
    uint2 pk;
    pk.x = pack_bf16x2(v.x, v.y);
    pk.y = pack_bf16x2(v.z, v.w);
    *reinterpret_cast<uint2*>(yr + c) = pk;
  }
}

__global__ void __launch_bounds__(256) embed_kernel(const bf16* __restrict__ wte, const bf16* __restrict__ wpe,
                                                    const int* __restrict__ tokens, const int* __restrict__ positions,
                                                    float* __restrict__ h, int d, int vocab, int n_pos) {
  ptx::grid_dep_wait();
  ptx::grid_dep_launch();
  const int r = blockIdx.x;
  // ids are range-checked by the host side (torch raises IndexError there); the clamp keeps a bad id handed to the C ABI
  // from becoming an illegal address that would poison the context
  const int tok = min(max(tokens[r], 0), vocab - 1);
  const uint2* te = reinterpret_cast<const uint2*>(wte + static_cast<long long>(tok) * d);
  const uint2* pe = wpe ? reinterpret_cast<const uint2*>(wpe + static_cast<long long>(min(max(positions[r], 0), n_pos - 1)) * d) : nullptr;
  float4* hr = reinterpret_cast<float4*>(h + static_cast<long long>(r) * d);
  for (int c = threadIdx.x; c < d / 4; c += blockDim.x) {
    const uint2 a = __ldg(te + c);
    float2 a0 = unpack_bf16x2(a.x), a1 = unpack_bf16x2(a.y);
    if (pe) {
      const uint2 p = __ldg(pe + c);
      const float2 p0 = unpack_bf16x2(p.x), p1 = unpack_bf16x2(p.y);
      a0.x += p0.x; a0.y += p0.y; a1.x += p1.x; a1.y += p1.y;
    }
    hr[c] = make_float4(a0.x, a0.y, a1.x, a1.y);
  }
}

__global__ void __launch_bounds__(256) add_positions_kernel(const float* __restrict__ src,
                                                            const bf16* __restrict__ wpe, int pos0, int S,
                                                            float* __restrict__ h, int d) {
  const int r = blockIdx.x;
  const int pos = pos0 + r % S;
  const float4* sr = reinterpret_cast<const float4*>(src + static_cast<long long>(r) * d);
  const uint2* pe = wpe ? reinterpret_cast<const uint2*>(wpe + static_cast<long long>(pos) * d) : nullptr;
  float4* hr = reinterpret_cast<float4*>(h + static_cast<long long>(r) * d);
  for (int c = threadIdx.x; c < d / 4; c += blockDim.x) {
    float4 v = sr[c];
    if (pe) {
      const uint2 p = __ldg(pe + c);
      const float2 p0 = unpack_bf16x2(p.x), p1 = unpack_bf16x2(p.y);
      v.x += p0.x; v.y += p0.y; v.z += p1.x; v.w += p1.y;
    }
    hr[c] = v;
  }
}

__global__ void __launch_bounds__(256) gather_rows_kernel(const float* __restrict__ src, long long lds, int gi, int go,
                                                          int off, float* __restrict__ dst, long long ldd, int d) {
  const int r = blockIdx.x;
  const long long sr = static_cast<long long>(r / gi) * go + off + r % gi;
  const float4* s4 = reinterpret_cast<const float4*>(src + sr * lds);
  float4* d4 = reinterpret_cast<float4*>(dst + static_cast<long long>(r) * ldd);
  for (int c = threadIdx.x; c < d / 4; c += blockDim.x) d4[c] = s4[c];
}

}  // namespace

int convert_rows_bf16(const void* src, int dtype, long long rows, int cols, bf16* dst, long long dst_ld,
                      cudaStream_t s) {
  if (rows <= 0 || cols <= 0) return 0;
  long long total = rows * cols;
  int blocks = static_cast<int>(total / 256 + 1 > 148 * 32 ? 148 * 32 : total / 256 + 1);
  if (dtype == 0)
    convert_rows_bf16_kernel<float><<<blocks, 256, 0, s>>>(static_cast<const float*>(src), rows, cols, dst, dst_ld);
  else if (dtype == 1)
    convert_rows_bf16_kernel<__half><<<blocks, 256, 0, s>>>(static_cast<const __half*>(src), rows, cols, dst, dst_ld);
  else if (dtype == 2)
    convert_rows_bf16_kernel<__nv_bfloat16><<<blocks, 256, 0, s>>>(static_cast<const __nv_bfloat16*>(src), rows, cols,
                                                                   dst, dst_ld);
  else
    return (int)cudaErrorInvalidValue;
  CCB_LAUNCH_CHECK();
  return 0;
}
int convert_f32(const void* src, int dtype, long long n, float* dst, cudaStream_t s) {
  if (n <= 0) return 0;
  int blocks = static_cast<int>(n / 256 + 1 > 148 * 32 ? 148 * 32 : n / 256 + 1);
  if (dtype == 0)
    convert_f32_kernel<float><<<blocks, 256, 0, s>>>(static_cast<const float*>(src), n, dst);
  else if (dtype == 1)
    convert_f32_kernel<__half><<<blocks, 256, 0, s>>>(static_cast<const __half*>(src), n, dst);
  else if (dtype == 2)
    convert_f32_kernel<__nv_bfloat16><<<blocks, 256, 0, s>>>(static_cast<const __nv_bfloat16*>(src), n, dst);
  else
    return (int)cudaErrorInvalidValue;
  CCB_LAUNCH_CHECK();
  return 0;
}
int transpose_bf16(const void* src, int dtype, int R, int C, bf16* dst, long long dst_ld, cudaStream_t s) {
  if (R <= 0 || C <= 0) return 0;
  dim3 grid((C + 31) / 32, (R + 31) / 32);
  if (dtype == 0)
    transpose_bf16_kernel<float><<<grid, 256, 0, s>>>(static_cast<const float*>(src), R, C, dst, dst_ld);
  else if (dtype == 1)
    transpose_bf16_kernel<__half><<<grid, 256, 0, s>>>(static_cast<const __half*>(src), R, C, dst, dst_ld);
  else if (dtype == 2)
    transpose_bf16_kernel<__nv_bfloat16><<<grid, 256, 0, s>>>(static_cast<const __nv_bfloat16*>(src), R, C, dst, dst_ld);
  else
    return (int)cudaErrorInvalidValue;
  CCB_LAUNCH_CHECK();
  return 0;
}

int layernorm_f32_bf16(const float* x, long long ldx, const float* gamma, const float* beta, float eps, bf16* y,
                       long long ldy, int rows, int d, cudaStream_t s) {
  if (rows <= 0) return 0;
  if (d % 4 || ldx % 4 || ldy % 4) return (int)cudaErrorInvalidValue;
  cudaError_t e;
  const int nq = d / 4;
  if (rows >= 256 && nq <= 32 * 32) {
    // many rows: one warp per row, 8 rows per CTA
    const dim3 grid((rows + 7) / 8), block(256);
    if (nq <= 32 * 8)
      e = launch_kernel(layernorm_rows_kernel<8>, grid, block, 0, s, true, x, ldx, gamma, beta, eps, y, ldy, rows, d);
    else if (nq <= 32 * 16)
      e = launch_kernel(layernorm_rows_kernel<16>, grid, block, 0, s, true, x, ldx, gamma, beta, eps, y, ldy, rows, d);
    else
      e = launch_kernel(layernorm_rows_kernel<32>, grid, block, 0, s, true, x, ldx, gamma, beta, eps, y, ldy, rows, d);
  } else {
    e = launch_kernel(layernorm_kernel<bf16>, dim3(rows), dim3(256), d * sizeof(float), s, true, x, ldx, gamma, beta, eps, y, ldy, d);
  }
  if (e != cudaSuccess) return (int)e;
  return 0;
}
int layernorm_f32_f32(const float* x, long long ldx, const float* gamma, const float* beta, float eps, float* y,
                      long long ldy, int rows, int d, cudaStream_t s) {
  if (rows <= 0) return 0;
  if (d % 4 || ldx % 4 || ldy % 4) return (int)cudaErrorInvalidValue;
  layernorm_kernel<float><<<rows, 256, d * sizeof(float), s>>>(x, ldx, gamma, beta, eps, y, ldy, d);
  CCB_LAUNCH_CHECK();
  return 0;
}

int vit_patchify(const void* images, int img_dtype, int B, int C, int H, int W, int ps, bf16* patches, int ldp,
                 cudaStream_t s) {
  if (B <= 0) return 0;
  if (ps <= 0 || H % ps || W % ps || ldp < C * ps * ps) return (int)cudaErrorInvalidValue;
  if (ps % 8 || ldp != C * ps * ps) {
    const long long total = static_cast<long long>(B) * (H / ps) * (W / ps) * ldp;
    int blocks = static_cast<int>((total + 255) / 256);
    if (blocks > 148 * 16) blocks = 148 * 16;
    if (img_dtype == 0)
      patchify_any_kernel<float><<<blocks, 256, 0, s>>>(static_cast<const float*>(images), B, C, H, W, ps, ldp, patches);
    else if (img_dtype == 1)
      patchify_any_kernel<__half><<<blocks, 256, 0, s>>>(static_cast<const __half*>(images), B, C, H, W, ps, ldp, patches);
    else if (img_dtype == 2)
      patchify_any_kernel<__nv_bfloat16><<<blocks, 256, 0, s>>>(static_cast<const __nv_bfloat16*>(images), B, C, H, W, ps, ldp,
                                                                patches);
    else
      return (int)cudaErrorInvalidValue;
    CCB_LAUNCH_CHECK();
    return 0;
  }
  const long long total8 = static_cast<long long>(B) * (H / ps) * (W / ps) * C * ps * ps / 8;
  int blocks = static_cast<int>((total8 + 255) / 256);
  if (blocks > 148 * 16) blocks = 148 * 16;
  if (img_dtype == 0)
    patchify_kernel<float><<<blocks, 256, 0, s>>>(static_cast<const float*>(images), B, C, H, W, ps, patches);
  else if (img_dtype == 1)
    patchify_kernel<__half><<<blocks, 256, 0, s>>>(static_cast<const __half*>(images), B, C, H, W, ps, patches);
  else if (img_dtype == 2)
    patchify_kernel<__nv_bfloat16><<<blocks, 256, 0, s>>>(static_cast<const __nv_bfloat16*>(images), B, C, H, W, ps,
                                                          patches);
  else
    return (int)cudaErrorInvalidValue;
  CCB_LAUNCH_CHECK();
  return 0;
}

int vit_assemble_lnpre(const float* patch_emb, const float* cls, const float* pos, const float* g, const float* b,
                       float eps, float* x, int B, int np, int d, cudaStream_t s) {
  if (B <= 0) return 0;
  vit_assemble_kernel<<<B * (np + 1), 256, d * sizeof(float), s>>>(patch_emb, cls, pos, g, b, eps, x, np, d);
  CCB_LAUNCH_CHECK();
  return 0;
}

int mapper_fill_const(const float* prefix_const, float* seq, int B, int clip_len, int P, int d, cudaStream_t s) {
  if (B <= 0 || P <= 0) return 0;
  if (d % 4) return (int)cudaErrorInvalidValue;
  mapper_fill_const_kernel<<<dim3(P, B), 256, 0, s>>>(prefix_const, seq, clip_len, P, d);
  CCB_LAUNCH_CHECK();
  return 0;
}

int mapper_fill_pos(const float* pos, float* seq, int B, int clip_len, int P, int d, cudaStream_t s) {
  if (B <= 0 || clip_len <= 0) return 0;
  if (d % 4) return (int)cudaErrorInvalidValue;
  mapper_fill_pos_kernel<<<dim3(clip_len, B), 256, 0, s>>>(pos, seq, clip_len, P, d);
  CCB_LAUNCH_CHECK();
  return 0;
}

// x, gate = chunk(2, -1); x * gelu(gate) with the erf form of nnf.gelu; one CTA per row, 8 bf16 per access
__global__ void geglu_kernel(bf16* __restrict__ x, long long ldx, int h) {
  bf16* row = x + static_cast<long long>(blockIdx.x) * ldx;
  for (int j = threadIdx.x * 8; j < h; j += blockDim.x * 8) {
    const uint4 a = *reinterpret_cast<const uint4*>(row + j), g = *reinterpret_cast<const uint4*>(row + h + j);
    const uint32_t av[4] = {a.x, a.y, a.z, a.w}, gv[4] = {g.x, g.y, g.z, g.w};
    uint32_t o[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float2 xa = unpack_bf16x2(av[k]), xg = unpack_bf16x2(gv[k]);
      o[k] = pack_bf16x2(xa.x * apply_act(xg.x, ACT_GELU_ERF), xa.y * apply_act(xg.y, ACT_GELU_ERF));
    }
    *reinterpret_cast<uint4*>(row + j) = make_uint4(o[0], o[1], o[2], o[3]);
  }
}

int geglu_inplace(bf16* x, long long ldx, int rows, int h, cudaStream_t s) {
  if (rows <= 0) return 0;
  if (h % 8 || ldx % 8) return (int)cudaErrorInvalidValue;
  geglu_kernel<<<rows, 256, 0, s>>>(x, ldx, h);
  CCB_LAUNCH_CHECK();
  return 0;
}

int cast_f32_bf16(const float* x, long long ldx, bf16* y, long long ldy, int rows, int d, cudaStream_t s) {
  if (rows <= 0) return 0;
  if (d % 4 || ldx % 4 || ldy % 4) return (int)cudaErrorInvalidValue;
  cast_kernel<<<rows, 256, 0, s>>>(x, ldx, y, ldy, d);
  CCB_LAUNCH_CHECK();
  return 0;
}

int embed_tokens(const bf16* wte, const bf16* wpe, const int* tokens, const int* positions, float* h, int rows, int d,
                 int vocab, int n_pos, cudaStream_t s) {
  if (rows <= 0) return 0;
  if (d % 4) return (int)cudaErrorInvalidValue;
  {
    cudaError_t e = launch_kernel(embed_kernel, dim3(rows), dim3(256), 0, s, true, wte, wpe, tokens, positions, h, d, vocab, n_pos);
    if (e != cudaSuccess) return (int)e;
  }
  return 0;
}

int add_positions(const float* src, const bf16* wpe, int pos0, int S, float* h, int rows, int d, cudaStream_t s) {
  if (rows <= 0) return 0;
  if (d % 4) return (int)cudaErrorInvalidValue;
  add_positions_kernel<<<rows, 256, 0, s>>>(src, wpe, pos0, S, h, d);
  CCB_LAUNCH_CHECK();
  return 0;
}

int gather_rows_f32(const float* src, long long lds, int gi, int go, int off, float* dst, long long ldd, int rows,
                    int d, cudaStream_t s) {
  if (rows <= 0) return 0;
  if (d % 4 || lds % 4 || ldd % 4) return (int)cudaErrorInvalidValue;
  gather_rows_kernel<<<rows, 256, 0, s>>>(src, lds, gi, go, off, dst, ldd, d);
  CCB_LAUNCH_CHECK();
  return 0;
}

bool pdl_enabled() {
  static const bool on = [] {
    const char* e = getenv("CCB_PDL");
    return !(e && e[0] == '0');
  }();
  return on;
}

}  // namespace ccb
