// On-device token selection: greedy arg-max, the reference's logit processors (repetition penalty, temperature,
// top-k, top-p; sampling.py:65-69,114-162 and inference.py:24-57) fused with softmax + multinomial sampling, the
// beam-search step of inference.py:98-131, and the per-step bookkeeping that lets the whole decode loop run
// without a host round-trip.
//
// Selection without sorting: the reference sorts all V logits to find the nucleus.  Here the boundary element
// is found with an 8-pass, 4-bit radix select over order-preserving float keys (per-thread private bins, so no
// shared-memory atomics), accumulating probability mass in double.  The kept set is identical to the
// reference's "sort, cumsum, shift-right" rule: an element is kept iff the mass of the elements ranked
// strictly before it is <= top_p (the first element crossing the threshold is kept, the top-1 always).
// When only the sampled token is asked for (top-p, no typical-p, no filtered logits, no second draw) the boundary is
// not needed at all: nucleus_sample_fast tests the best few candidates of argmax(p / q) for membership with that rule
// and falls back to the select on a miss or a near-tie.
// The beam step is two launches: beam_rows_kernel (one CTA per (image, beam row): the row's candidates) and
// beam_merge_kernel (one CTA per image: merge, bookkeeping, block-table permutation).
#include <float.h>

#include "common.cuh"
#include "internal.h"
#include "ptx.cuh"

namespace ccb {

namespace {

constexpr int kSampThreads = 1024;

__device__ __forceinline__ uint32_t order_key(float x) {
  const uint32_t u = __float_as_uint(x);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// Philox4x32-10 (Salmon et al.), the counter-based generator used when no explicit noise tensor is given.
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(M0, ctr.x), lo0 = M0 * ctr.x;
    const uint32_t hi1 = __umulhi(M1, ctr.z), lo1 = M1 * ctr.z;
    ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
    key.x += W0;
    key.y += W1;
  }
  return ctr;
}
// the four Exp(1) values of elements 4 g .. 4 g + 3 (one Philox call; identical to philox_exp1 of each element)
__device__ __forceinline__ float4 philox_exp1_x4(unsigned long long seed, unsigned long long row, uint32_t step, uint32_t g) {
  const uint4 c = make_uint4(g, step, static_cast<uint32_t>(row), static_cast<uint32_t>(row >> 32));
  const uint2 k = make_uint2(static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32));
  const uint4 r = philox4x32_10(c, k);
  const float sc = 1.0f / 16777216.0f;
  return make_float4(-logf((static_cast<float>(r.x >> 8) + 0.5f) * sc), -logf((static_cast<float>(r.y >> 8) + 0.5f) * sc),
                     -logf((static_cast<float>(r.z >> 8) + 0.5f) * sc), -logf((static_cast<float>(r.w >> 8) + 0.5f) * sc));
}
__device__ __forceinline__ float philox_exp1(unsigned long long seed, unsigned long long row, uint32_t step,
                                             uint32_t v) {
  const uint4 c = make_uint4(v >> 2, step, static_cast<uint32_t>(row), static_cast<uint32_t>(row >> 32));
  const uint2 k = make_uint2(static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32));
  const uint4 r = philox4x32_10(c, k);
  const uint32_t w = (v & 3) == 0 ? r.x : (v & 3) == 1 ? r.y : (v & 3) == 2 ? r.z : r.w;
  const float u = (static_cast<float>(w >> 8) + 0.5f) * (1.0f / 16777216.0f);  // (0,1)
  return -logf(u);
}

struct ArgMax {
  float v;
  int i;
};
__device__ __forceinline__ ArgMax argmax_better(ArgMax a, ArgMax b) {
  // larger value wins; equal values -> lower index wins
  if (b.v > a.v || (b.v == a.v && b.i < a.i)) return b;
  return a;
}
__device__ __forceinline__ ArgMax block_argmax(ArgMax a, ArgMax* scratch /*>=32*/) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ArgMax b;
    b.v = __shfl_xor_sync(0xffffffffu, a.v, o);
    b.i = __shfl_xor_sync(0xffffffffu, a.i, o);
    a = argmax_better(a, b);
  }
  __syncthreads();
  if (lane == 0) scratch[w] = a;
  __syncthreads();
  ArgMax r;
  r.v = -INFINITY;
  r.i = 0x7fffffff;
  if (lane < nw) r = scratch[lane];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ArgMax b;
    b.v = __shfl_xor_sync(0xffffffffu, r.v, o);
    b.i = __shfl_xor_sync(0xffffffffu, r.i, o);
    r = argmax_better(r, b);
  }
  return r;
}

__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double block_sum_d(double v, double* scratch /*>=32*/) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  v = warp_sum_d(v);
  __syncthreads();
  if (lane == 0) scratch[w] = v;
  __syncthreads();
  double r = (lane < nw) ? scratch[lane] : 0.0;
  return warp_sum_d(r);
}
__device__ __forceinline__ int block_sum_i(int v, int* scratch) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  __syncthreads();
  if (lane == 0) scratch[w] = v;
  __syncthreads();
  int r = (lane < nw) ? scratch[lane] : 0;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) r += __shfl_xor_sync(0xffffffffu, r, o);
  return r;
}

// ------------------------------------------------------------------------------------------------ greedy
__global__ void __launch_bounds__(kSampThreads) greedy_kernel(const float* __restrict__ logits, long long ld, int V,
                                                              int* __restrict__ next) {
  __shared__ ArgMax scratch[32];
  ptx::grid_dep_wait();
  ptx::grid_dep_launch();
  const float* row = logits + static_cast<long long>(blockIdx.x) * ld;
  ArgMax a;
  a.v = -INFINITY;
  a.i = 0x7fffffff;
  int v_done = 0;
  if ((reinterpret_cast<uintptr_t>(row) & 15) == 0) {
    // 16-byte loads, four per thread in flight (one row = 50 257 floats on 1024 threads: 12.3 float4 per thread)
    const float4* row4 = reinterpret_cast<const float4*>(row);
    const int nq = V >> 2;
    for (int q0 = threadIdx.x; q0 < nq; q0 += 4 * kSampThreads) {
      float4 w[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int q = q0 + j * kSampThreads;
        w[j] = q < nq ? row4[q] : make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int q = q0 + j * kSampThreads;
        if (q >= nq) continue;
        const float e[4] = {w[j].x, w[j].y, w[j].z, w[j].w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          ArgMax b;
          b.v = e[k];
          b.i = 4 * q + k;
          a = argmax_better(a, b);
        }
      }
    }
    v_done = nq << 2;
  }
  for (int v = v_done + threadIdx.x; v < V; v += blockDim.x) {
    ArgMax b;
    b.v = row[v];
    b.i = v;
    a = argmax_better(a, b);
  }
  a = block_argmax(a, scratch);
  if (threadIdx.x == 0) next[blockIdx.x] = a.i;
}

// ------------------------------------------------------------------------------------------------ cross entropy
// F.cross_entropy(logits.reshape(-1, V), targets, ignore_index) of evaluate_model.py:511-514 / model.py:210-211 (the
// teacher-forced validation / training loss).  One CTA per target row: max, log-sum-exp (sum in double), minus the target's
// logit; rows whose target is ignore_index give 0 and are not counted.  row_map (optional) = index of the logits row of
// each target, so the reference's `logits[:, P-1:-1]` slice needs no copy.
__global__ void __launch_bounds__(kSampThreads) cross_entropy_rows_kernel(const float* __restrict__ logits, long long ld, int V,
                                                                          const int* __restrict__ targets, const int* __restrict__ row_map,
                                                                          int ignore_index, float* __restrict__ row_loss) {
  __shared__ ArgMax ascratch[32];
  __shared__ double dscratch[32];
  const int r = blockIdx.x;
  const int tgt = targets[r];
  if (tgt == ignore_index || tgt < 0 || tgt >= V) {   // (out-of-range targets other than ignore_index are an error in torch; host-checked)
    if (threadIdx.x == 0) row_loss[r] = 0.f;
    return;
  }
  const float* row = logits + static_cast<long long>(row_map ? row_map[r] : r) * ld;
  ArgMax a;
  a.v = -INFINITY;
  a.i = 0x7fffffff;
  for (int v = threadIdx.x; v < V; v += kSampThreads) {
    ArgMax b;
    b.v = row[v];
    b.i = v;
    a = argmax_better(a, b);
  }
  a = block_argmax(a, ascratch);
  const float vmax = a.v;
  double sum = 0.0;
  for (int v = threadIdx.x; v < V; v += kSampThreads) sum += static_cast<double>(expf(row[v] - vmax));
  sum = block_sum_d(sum, dscratch);
  if (threadIdx.x == 0) row_loss[r] = static_cast<float>(static_cast<double>(vmax) + log(sum) - static_cast<double>(row[tgt]));
}

// mean over the counted rows, summed in row order by one CTA (deterministic); out = {mean, count}
__global__ void __launch_bounds__(kSampThreads) cross_entropy_mean_kernel(const float* __restrict__ row_loss, const int* __restrict__ targets,
                                                                          int rows, int ignore_index, float* __restrict__ out) {
  __shared__ double dscratch[32];
  __shared__ int iscratch[32];
  double s = 0.0;
  int n = 0;
  for (int r = threadIdx.x; r < rows; r += kSampThreads) {
    if (targets[r] != ignore_index) {
      s += static_cast<double>(row_loss[r]);
      ++n;
    }
  }
  s = block_sum_d(s, dscratch);
  n = block_sum_i(n, iscratch);
  if (threadIdx.x == 0) {
    out[0] = static_cast<float>(s / static_cast<double>(n));   // 0 / 0 = NaN, as torch
    out[1] = static_cast<float>(n);
  }
}

// ------------------------------------------------------------------------------------------------ top-k / top-p
// 4-bit radix select over the order keys of vals[0..V).  mode 0: k-th largest (by count, 1-based `kth`).
// mode 1: first element (descending) at which the cumulative probability mass exceeds top_p, where the mass of
// element i is expf(vals[i] - vmax) * inv_sum.  mode 2 (typical decoding, sampling.py:72-102): the elements are ordered by
// ASCENDING |log p_i + H| (log p_i = vals[i] - vmax - lse, H the entropy) and the boundary is the first element at which
// the cumulative probability is no longer below top_p.  Returns through shared scalars:
//   sel_key  : key of the boundary element (0 when the target is never reached -> keep everything)
//   mass_gt  : mode 1: mass strictly above the boundary key;   cnt_eq: elements equal to the boundary key
struct SelectResult {
  uint32_t key;
  double mass_gt;
  int cnt_eq;
  int reached;
};

__device__ __forceinline__ uint32_t typical_key(float x, float vmax, float lse, float ent) {
  return order_key(-fabsf(((x - vmax) - lse) + ent));   // descending key order == ascending distance to the entropy
}

__device__ SelectResult radix_select(const float* vals, int V, int mode, int kth, float top_p, float vmax,
                                     float inv_sum, double* dscratch /*32 + 16*/, int* iscratch /*32 + 16*/,
                                     float lse = 0.f, float ent = 0.f) {
  uint32_t prefix = 0;
  double mass_above = 0.0;
  int cnt_above = 0;
  int reached = 1;
  int cnt_eq = 0;
  double* bin_mass = dscratch + 32;
  int* bin_cnt = iscratch + 32;
  for (int nib = 7; nib >= 0; --nib) {
    const int shift = nib * 4;
    double m[16];
    int c[16];
#pragma unroll
    for (int b = 0; b < 16; ++b) {
      m[b] = 0.0;
      c[b] = 0;
    }
    for (int v = threadIdx.x; v < V; v += blockDim.x) {
      const float x = vals[v];
      const uint32_t key = mode == 2 ? typical_key(x, vmax, lse, ent) : order_key(x);
      const bool match = (nib == 7) || ((key >> (shift + 4)) == (prefix >> (shift + 4)));
      if (match) {
        const int b = (key >> shift) & 15;
        double pm = 0.0;
        if (mode == 1) pm = static_cast<double>(expf(x - vmax) * inv_sum);
        if (mode == 2) pm = static_cast<double>(expf((x - vmax) - lse));
#pragma unroll
        for (int q = 0; q < 16; ++q) {
          if (q == b) {
            m[q] += pm;
            c[q] += 1;
          }
        }
      }
    }
    // the 16 (count, mass) pairs of all threads -> block totals with ONE pair of CTA barriers: shuffle tree inside a
    // warp, then thread b adds the warps' totals of bin b in warp order (a fixed order: deterministic masses)
    {
      __shared__ int warp_cnt[32][16];
      __shared__ double warp_mass[32][16];
      const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
#pragma unroll
      for (int b = 0; b < 16; ++b) {
        int cb = c[b];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) cb += __shfl_xor_sync(0xffffffffu, cb, o);
        double mb = 0.0;
        if (mode != 0) mb = warp_sum_d(m[b]);
        if (lane == 0) {
          warp_cnt[w][b] = cb;
          warp_mass[w][b] = mb;
        }
      }
      __syncthreads();
      if (threadIdx.x < 16) {
        int cb = 0;
        double mb = 0.0;
        for (int ww = 0; ww < nw; ++ww) {
          cb += warp_cnt[ww][threadIdx.x];
          mb += warp_mass[ww][threadIdx.x];
        }
        bin_cnt[threadIdx.x] = cb;
        bin_mass[threadIdx.x] = mb;
      }
    }
    __syncthreads();
    // every thread scans the 16 totals identically
    int chosen = -1;
    for (int b = 15; b >= 0; --b) {
      if (bin_cnt[b] == 0) continue;
      bool hit;
      if (mode == 0)
        hit = (cnt_above + bin_cnt[b] >= kth);
      else if (mode == 1)
        hit = (static_cast<float>(mass_above + bin_mass[b]) > top_p);
      else
        hit = !(static_cast<float>(mass_above + bin_mass[b]) < top_p);
      if (hit) {
        chosen = b;
        break;
      }
      cnt_above += bin_cnt[b];
      mass_above += bin_mass[b];
    }
    if (chosen < 0) {
      reached = 0;
      break;
    }
    prefix |= static_cast<uint32_t>(chosen) << shift;
    cnt_eq = bin_cnt[chosen];
    __syncthreads();
  }
  __syncthreads();
  SelectResult r;
  r.key = reached ? prefix : 0u;
  r.mass_gt = mass_above;
  r.cnt_eq = cnt_eq;
  r.reached = reached;
  return r;
}

struct TopPArgs {
  const float* logits;
  long long ld;
  int V;
  float temperature;
  float top_p;
  int top_k;
  const float* top_p_rows;
  const int* top_k_rows;
  float typ_p;
  const float* typ_p_rows;
  float rep_pen;
  const int* history;
  long long ld_hist;
  const int* hist_len;
  int hist_len_scalar;
  int hist_len_from_step;
  const float* q_noise;
  long long ldq;
  long long q_step_stride;
  unsigned long long seed;
  const long long* row_ids;
  const int* step;
  int step_scalar;
  const int* row_step;
  float* filtered_out;
  int* alt_out;
  int* next;
  int fast;   // 1: try nucleus_sample_fast first
};


// ---- sampling from the nucleus WITHOUT finding its boundary (the common case: top-p only, nothing but the token asked for)
// multinomial(softmax(filtered)) == argmax over the kept set S of p_v / q_v, and dividing by the kept mass does not change
// the arg-max.  So: rank all tokens by r'_v = exp(x_v - max) / q_v, take the best few, and test them for membership in S in
// that order -- "v is kept iff the probability mass ranked strictly before it is <= top_p" (see the header comment) is ONE
// masked sum over the row, not a selection.  The first candidate inside S is the sample; it is accepted only if it leads the
// next-ranked candidate by more than the rounding the exact path's extra division (p / kept_mass) could introduce (1e-6
// relative, two fp32 roundings are 1.2e-7), so the result is the exact path's token, ties included.  Everything else --
// no candidate in S among the first six (probability (1 - top_p)^6), a near-tie, a thread holding more than four of the
// top seven -- falls through to the radix select below.  5 light passes over the row instead of 8 heavy ones + 2.
struct Top4 {
  float v[4];
  int i[4];
};
__device__ __forceinline__ void top4_insert(Top4& t, float v, int i) {
  // (v, i) ranks before (tv, ti) iff v > tv or (v == tv and i < ti)
  if (!(v > t.v[3] || (v == t.v[3] && i < t.i[3]))) return;
  int pos = 3;
#pragma unroll
  for (int k = 2; k >= 0; --k)
    if (v > t.v[k] || (v == t.v[k] && i < t.i[k])) pos = k;
#pragma unroll
  for (int k = 3; k > 0; --k)
    if (k > pos) { t.v[k] = t.v[k - 1]; t.i[k] = t.i[k - 1]; }
#pragma unroll
  for (int k = 0; k < 4; ++k)
    if (k == pos) { t.v[k] = v; t.i[k] = i; }
}

// returns the sampled token or -1 (block-uniform) when the exact path has to decide
__device__ int nucleus_sample_fast(const float* vals, int V, float mx, float inv_sum, float top_p, const float* qrow,
                                   unsigned long long seed, unsigned long long rid, uint32_t step, ArgMax* ascratch,
                                   double* dscratch, int* iscratch) {
  constexpr int NC = 7;   // candidates: six testable + one more for the last one's margin
  Top4 loc;
#pragma unroll
  for (int k = 0; k < 4; ++k) { loc.v[k] = -INFINITY; loc.i[k] = 0x7fffffff; }
  int seen = 0;
  if (qrow != nullptr) {
    for (int v = threadIdx.x; v < V; v += blockDim.x) {
      const float x = vals[v];
      if (x == -INFINITY) continue;
      ++seen;
      top4_insert(loc, expf(x - mx) / qrow[v], v);
    }
  } else {
    for (int g = threadIdx.x; 4 * g < V; g += blockDim.x) {
      float x[4];
      bool any = false;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        x[k] = (4 * g + k < V) ? vals[4 * g + k] : -INFINITY;
        any |= x[k] != -INFINITY;
      }
      if (!any) continue;
      const float4 q4 = philox_exp1_x4(seed, rid, step, static_cast<uint32_t>(g));
      const float q[4] = {q4.x, q4.y, q4.z, q4.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        if (x[k] == -INFINITY) continue;
        ++seen;
        top4_insert(loc, expf(x[k] - mx) / q[k], 4 * g + k);
      }
    }
  }
  // the block's best NC, in rank order: NC arg-max rounds, the owner of a winner pops it
  float cv[NC];
  int ci[NC];
  int popped = 0;
#pragma unroll
  for (int j = 0; j < NC; ++j) {
    ArgMax mine;
    mine.v = loc.v[0];
    mine.i = loc.i[0];
    const ArgMax win = block_argmax(mine, ascratch);
    cv[j] = win.v;
    ci[j] = win.i;
    if (win.i == loc.i[0] && loc.i[0] != 0x7fffffff) {
#pragma unroll
      for (int k = 0; k < 3; ++k) { loc.v[k] = loc.v[k + 1]; loc.i[k] = loc.i[k + 1]; }
      loc.v[3] = -INFINITY;
      loc.i[3] = 0x7fffffff;
      ++popped;
    }
  }
  // a thread that gave all four of its entries away may hold a better fifth than what the block saw
  if (__syncthreads_or(popped == 4 && seen > 4)) return -1;
#pragma unroll 1
  for (int j = 0; j + 1 < NC; j += 2) {
    const int ia = ci[j], ib = ci[j + 1];
    if (ia == 0x7fffffff) return -1;                  // fewer candidates than that: nothing left to test
    const bool has_b = ib != 0x7fffffff;
    const float xa = vals[ia], xb = has_b ? vals[ib] : 0.f;
    const uint32_t ka = order_key(xa), kb = has_b ? order_key(xb) : 0xffffffffu;
    const uint32_t klo = ka < kb ? ka : kb;
    double ma = 0.0, mb = 0.0;
    int ta = 0, tb = 0;
    for (int v = threadIdx.x; v < V; v += blockDim.x) {
      const float x = vals[v];
      const uint32_t key = order_key(x);
      if (key < klo) continue;
      const double pm = static_cast<double>(expf(x - mx) * inv_sum);
      if (key > ka) ma += pm;
      else if (key == ka && v < ia) ++ta;
      if (key > kb) mb += pm;
      else if (key == kb && v < ib) ++tb;
    }
    ma = block_sum_d(ma, dscratch);
    mb = block_sum_d(mb, dscratch);
    ta = block_sum_i(ta, iscratch);
    tb = block_sum_i(tb, iscratch);
    const double pa = static_cast<double>(expf(xa - mx) * inv_sum), pb = static_cast<double>(expf(xb - mx) * inv_sum);
    const bool in_a = !(static_cast<float>(ma + ta * pa) > top_p);
    const bool in_b = has_b && !(static_cast<float>(mb + tb * pb) > top_p);
    // (exp(x - max) > 1e-20 keeps p = exp / kept_mass a normal number, so the relative rounding bound above holds)
    if (in_a) return (expf(xa - mx) > 1e-20f && cv[j] > cv[j + 1] * 1.000001f) ? ia : -1;
    if (in_b) return (j + 2 < NC && expf(xb - mx) > 1e-20f && cv[j + 1] > cv[j + 2] * 1.000001f) ? ib : -1;
  }
  return -1;
}

__global__ void __launch_bounds__(kSampThreads) top_p_kernel(const TopPArgs a) {
  extern __shared__ float vals[];  // V floats
  __shared__ double dscratch[48];
  __shared__ int iscratch[48];
  __shared__ ArgMax ascratch[32];
  __shared__ float fscratch[32];
  const int b = blockIdx.x;
  const int V = a.V;
  const float* row = a.logits + static_cast<long long>(b) * a.ld;

  // the row into shared memory: 16-byte cp.async copies, all of a thread's ~12 in flight at once (a scalar load -> store
  // loop keeps one or two L2 round trips in flight per thread and took 26 of the kernel's 90 us at 1024 threads)
  if ((reinterpret_cast<uintptr_t>(row) & 15) == 0) {
    const uint32_t vals_u32 = ptx::smem_u32(vals);
    const int nq = V >> 2;
    for (int q = threadIdx.x; q < nq; q += blockDim.x)
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(vals_u32 + 16u * q), "l"(row + 4 * q) : "memory");
    asm volatile("cp.async.commit_group;" ::: "memory");
    for (int v = 4 * nq + threadIdx.x; v < V; v += blockDim.x) vals[v] = row[v];
    asm volatile("cp.async.wait_group 0;" ::: "memory");
  } else {
    for (int v = threadIdx.x; v < V; v += blockDim.x) vals[v] = row[v];
  }
  __syncthreads();
  // repetition penalty (values computed from the ORIGINAL logits, like gather -> where -> scatter_)
  if (a.rep_pen != 1.0f && a.history != nullptr) {
    const int hl = a.row_step ? a.row_step[b]
                 : a.hist_len ? a.hist_len[b] : (a.hist_len_from_step && a.step ? *a.step : a.hist_len_scalar);
    for (int t = threadIdx.x; t < hl; t += blockDim.x) {
      const int tok = a.history[static_cast<long long>(b) * a.ld_hist + t];
      if (tok >= 0 && tok < V) {
        const float x = row[tok];
        vals[tok] = (x < 0.f) ? x * a.rep_pen : x / a.rep_pen;
      }
    }
    __syncthreads();
  }
  const float T = a.temperature > 0.f ? a.temperature : 1.0f;
  if (T != 1.0f) {
    for (int v = threadIdx.x; v < V; v += blockDim.x) vals[v] = vals[v] / T;
    __syncthreads();
  }

  // ---- top-k: remove everything strictly below the k-th largest value (ties at the cutoff survive)
  int k = a.top_k_rows ? a.top_k_rows[b] : a.top_k;
  if (k > V) k = V;
  if (k > 0) {
    const SelectResult r = radix_select(vals, V, 0, k, 0.f, 0.f, 0.f, dscratch, iscratch);
    for (int v = threadIdx.x; v < V; v += blockDim.x)
      if (order_key(vals[v]) < r.key) vals[v] = -INFINITY;
    __syncthreads();
  }

  // ---- row max and softmax denominator of the (top-k filtered) row
  float mx = -INFINITY;
  for (int v = threadIdx.x; v < V; v += blockDim.x) mx = fmaxf(mx, vals[v]);
  mx = block_max(mx, fscratch);
  float sum = 0.f;
  for (int v = threadIdx.x; v < V; v += blockDim.x) sum += expf(vals[v] - mx);
  sum = block_sum(sum, fscratch);

  // ---- top-p
  const float top_p = a.top_p_rows ? a.top_p_rows[b] : a.top_p;
  {
    const float typ = a.typ_p_rows ? a.typ_p_rows[b] : a.typ_p;
    const bool typ_on = (a.typ_p_rows != nullptr && typ >= 0.f) || (a.typ_p_rows == nullptr && typ > 0.f);
    if (a.fast && top_p > 0.f && !typ_on && a.filtered_out == nullptr && a.alt_out == nullptr) {
      const unsigned long long rid_f = a.row_ids ? static_cast<unsigned long long>(a.row_ids[b]) : static_cast<unsigned long long>(b);
      const uint32_t step_f = a.row_step ? static_cast<uint32_t>(a.row_step[b])
                            : a.step ? static_cast<uint32_t>(*a.step) : static_cast<uint32_t>(a.step_scalar);
      const float* qrow_f = a.q_noise ? a.q_noise + static_cast<long long>(step_f) * a.q_step_stride + static_cast<long long>(b) * a.ldq : nullptr;
      const int tok = nucleus_sample_fast(vals, V, mx, 1.0f / sum, top_p, qrow_f, a.seed, rid_f, step_f, ascratch, dscratch, iscratch);
      if (tok >= 0) {
        if (threadIdx.x == 0) a.next[b] = tok;
        return;
      }
    }
  }
  if (top_p > 0.f) {
    const SelectResult r = radix_select(vals, V, 1, 0, top_p, mx, 1.0f / sum, dscratch, iscratch);
    if (r.reached) {
      // how many of the elements equal to the boundary key are kept (usually exactly one)
      int keep_eq = r.cnt_eq;
      if (r.cnt_eq > 1) {
        // boundary probability: all ties share it
        float xb = 0.f;
        {
          const uint32_t kk = r.key;
          const uint32_t u = (kk & 0x80000000u) ? (kk & 0x7fffffffu) : ~kk;
          xb = __uint_as_float(u);
        }
        const double pb = static_cast<double>(expf(xb - mx) * (1.0f / sum));
        keep_eq = 1;
        while (keep_eq < r.cnt_eq && !(static_cast<float>(r.mass_gt + keep_eq * pb) > top_p)) ++keep_eq;
      }
      if (keep_eq >= r.cnt_eq) {
        for (int v = threadIdx.x; v < V; v += blockDim.x)
          if (order_key(vals[v]) < r.key) vals[v] = -INFINITY;
      } else {
        // rare: keep only the first keep_eq ties in index order -> blocked ranges + block scan of tie counts
        const int per = (V + blockDim.x - 1) / blockDim.x;
        const int lo = threadIdx.x * per, hi = min(V, lo + per);
        int mine = 0;
        for (int v = lo; v < hi; ++v) mine += (order_key(vals[v]) == r.key);
        __shared__ int tie_prefix[kSampThreads];
        tie_prefix[threadIdx.x] = mine;
        __syncthreads();
        if (threadIdx.x == 0) {
          int run = 0;
          for (int t = 0; t < blockDim.x; ++t) {
            const int c = tie_prefix[t];
            tie_prefix[t] = run;
            run += c;
          }
        }
        __syncthreads();
        int rank = tie_prefix[threadIdx.x];
        for (int v = lo; v < hi; ++v) {
          const uint32_t key = order_key(vals[v]);
          if (key < r.key) {
            vals[v] = -INFINITY;
          } else if (key == r.key) {
            if (rank >= keep_eq) vals[v] = -INFINITY;
            ++rank;
          }
        }
      }
      __syncthreads();
    }
  }
  // ---- typical filtering (sampling.py:72-102), on the row as filtered so far (sampling.py:205-206)
  // (per-row budgets: every row is filtered, a budget of 0 keeps the most typical token, as in the reference when some
  //  budget is positive; a NEGATIVE budget is this library's "leave the row alone" -- the device-side loop of
  //  clipcap_b200.sampling.generate uses it when no active row has a positive budget)
  const float typ_p = a.typ_p_rows ? a.typ_p_rows[b] : a.typ_p;
  if ((a.typ_p_rows != nullptr && typ_p >= 0.f) || (a.typ_p_rows == nullptr && typ_p > 0.f)) {
    float s2 = 0.f;
    for (int v = threadIdx.x; v < V; v += blockDim.x) s2 += expf(vals[v] - mx);
    s2 = block_sum(s2, fscratch);
    const float lse = logf(s2);
    float e = 0.f;
    for (int v = threadIdx.x; v < V; v += blockDim.x) {
      const float x = vals[v];
      if (x != -INFINITY) {
        const float lp = (x - mx) - lse;
        e += lp * expf(lp);
      }
    }
    const float ent = -block_sum(e, fscratch);
    const SelectResult r = radix_select(vals, V, 2, 0, typ_p, mx, 0.f, dscratch, iscratch, lse, ent);
    if (r.reached) {
      for (int v = threadIdx.x; v < V; v += blockDim.x)
        if (typical_key(vals[v], mx, lse, ent) < r.key) vals[v] = -INFINITY;
      __syncthreads();
    }
  }
  if (a.filtered_out) {
    float* fo = a.filtered_out + static_cast<long long>(b) * a.ld;
    for (int v = threadIdx.x; v < V; v += blockDim.x) fo[v] = vals[v];
  }

  // ---- softmax over the kept set and multinomial == argmax(p / q), q ~ Exp(1)
  float ksum = 0.f;
  for (int v = threadIdx.x; v < V; v += blockDim.x) ksum += expf(vals[v] - mx);
  ksum = block_sum(ksum, fscratch);
  const unsigned long long rid = a.row_ids ? static_cast<unsigned long long>(a.row_ids[b]) : static_cast<unsigned long long>(b);
  const uint32_t step = a.row_step ? static_cast<uint32_t>(a.row_step[b])
                      : a.step ? static_cast<uint32_t>(*a.step) : static_cast<uint32_t>(a.step_scalar);
  const float* qrow = a.q_noise ? a.q_noise + static_cast<long long>(step) * a.q_step_stride + static_cast<long long>(b) * a.ldq : nullptr;
  ArgMax best;
  best.v = -INFINITY;
  best.i = 0x7fffffff;
  if (qrow != nullptr) {
    for (int v = threadIdx.x; v < V; v += blockDim.x) {
      const float x = vals[v];
      if (x == -INFINITY) continue;
      const float p = expf(x - mx) / ksum;
      ArgMax c;
      c.v = p / qrow[v];
      c.i = v;
      best = argmax_better(best, c);
    }
  } else {
    // a thread takes the four elements that share one Philox block (the noise of element v is word v & 3 of block v >> 2)
    for (int g = threadIdx.x; 4 * g < V; g += blockDim.x) {
      float x[4];
      bool any = false;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        x[k] = (4 * g + k < V) ? vals[4 * g + k] : -INFINITY;
        any |= x[k] != -INFINITY;
      }
      if (!any) continue;
      const float4 q4 = philox_exp1_x4(a.seed, rid, step, static_cast<uint32_t>(g));
      const float q[4] = {q4.x, q4.y, q4.z, q4.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        if (x[k] == -INFINITY) continue;
        ArgMax c;
        c.v = (expf(x[k] - mx) / ksum) / q[k];
        c.i = 4 * g + k;
        best = argmax_better(best, c);
      }
    }
  }
  const ArgMax win = block_argmax(best, ascratch);
  if (threadIdx.x == 0) a.next[b] = win.i;
  if (a.alt_out) {
    // second draw without replacement: best ratio excluding the winner
    ArgMax second;
    second.v = -INFINITY;
    second.i = 0x7fffffff;
    for (int v = threadIdx.x; v < V; v += blockDim.x) {
      const float x = vals[v];
      if (x == -INFINITY || v == win.i) continue;
      const float p = expf(x - mx) / ksum;
      const float q = qrow ? qrow[v] : philox_exp1(a.seed, rid, step, v);
      ArgMax c;
      c.v = p / q;
      c.i = v;
      second = argmax_better(second, c);
    }
    const ArgMax w2 = block_argmax(second, ascratch);
    if (threadIdx.x == 0) a.alt_out[b] = (w2.i == 0x7fffffff) ? win.i : w2.i;
  }
}

// ------------------------------------------------------------------------------------------------ beam step
// One CTA per image.  Follows inference.py:98-131 (see SURVEY appendix A.4):
//   lp = log(softmax(logits / T));  first step: scores, tokens = top-beam(lp[row 0])
//   later: stopped rows contribute only token 0 with lp 0; sum = score + lp; len += !stopped; avg = sum / len;
//          flat top-beam over beam*V of avg (ties: lowest flat index); src = idx / V; tok = idx % V;
//          len = len[src]; score = avg * len; stopped = stopped[src] | (tok == stop)
// Also permutes the per-row token history and block tables so the next decode step reads the right KV.
constexpr int kMaxBeam = 8;
static_assert(kMaxBeam == kBeamCandPerRow, "candidate scratch rows are sized by internal.h");

struct Cand {
  float v;
  int idx;  // flat index r * V + tok
};
__device__ __forceinline__ bool cand_better(const Cand& a, const Cand& b) {  // a ranks before b
  return a.v > b.v || (a.v == b.v && a.idx < b.idx);
}

struct BeamArgs {
  Cand* cand;               // [N*beam, kMaxBeam] the rows' best candidates (beam_rows_kernel -> beam_merge_kernel)
  const float* logits;      // step 0: [N, ld] (one row per image); later: [N*beam, ld]
  long long ld;
  int beam, V;
  float temperature;
  int stop_token;
  float* scores;
  float* seq_lengths;
  uint8_t* has_stopped;
  int* tokens;              // [N, beam, max_len]
  int max_len;
  const int* step;
  int* next_tokens;         // [N*beam]
  int* src_rows;            // [N*beam]
  int* block_table;         // [N*beam, max_pages] permuted in place (may be null)
  int max_pages;
  int* ctx_len;             // [N*beam] tokens currently cached per row (entries < ctx are permuted)
  BeamGroups grp;           // per-group mode (internal.h) when grp.group_step is non-null
};

// group of launch entry n in per-group mode (the entry itself otherwise); true when that group is frozen
__device__ __forceinline__ bool beam_group(const BeamArgs& a, int n, int& g) {
  g = a.grp.slots ? a.grp.slots[n] : n;
  return a.grp.group_step && (a.grp.group_image[g] < 0 || a.grp.finished[g]);
}

// Two launches per step.  beam_rows_kernel: one CTA per (image, beam row) -- the row's log-softmax statistics and its
// best kMaxBeam candidates (255 rows keep every SM busy where one CTA per image used 51 of 148).  beam_merge_kernel: one
// CTA per image merges the rows' candidate lists (the top-beam of the union is the top-beam of the union of the rows'
// top-beams) and does the bookkeeping.
constexpr int kBeamRowThreads = 512;

__global__ void __launch_bounds__(kBeamRowThreads, 2) beam_rows_kernel(const BeamArgs a) {
  __shared__ float fscratch[32];
  __shared__ Cand wcand[(kBeamRowThreads / 32) * kMaxBeam];
  const int beam = a.beam, V = a.V;
  const int n = blockIdx.x / beam, r = blockIdx.x - n * beam;
  int g;
  if (beam_group(a, n, g)) return;
  const int step = a.grp.group_step ? a.grp.group_step[g] : *a.step;
  const bool first = (step == 0);
  if (first && r > 0) return;          // the first step ranks the single prefill row of the image
  Cand* out = a.cand + static_cast<long long>(blockIdx.x) * kMaxBeam;
  const float T = a.temperature > 0.f ? a.temperature : 1.0f;
  const bool unit_T = T == 1.0f;       // x / 1.0f == x: skip the division
  const float score = first ? 0.f : a.scores[g * beam + r];
  const bool stopped = !first && a.has_stopped[g * beam + r];
  // seq_lengths[~has_stopped] += 1  (not on the first step)
  const float len = first ? 1.f : a.seq_lengths[g * beam + r] + (stopped ? 0.f : 1.f);
  if (stopped) {
    // logits[has_stopped] = -inf; logits[has_stopped, 0] = 0  -> only token 0 is a finite candidate
    if (threadIdx.x < kMaxBeam) {
      Cand c;
      c.v = threadIdx.x == 0 ? (score + 0.f) / len : -INFINITY;
      c.idx = threadIdx.x == 0 ? r * V : 0x7fffffff;
      out[threadIdx.x] = c;
    }
    return;
  }
  const float* row = a.logits + (first ? static_cast<long long>(n) : static_cast<long long>(n) * beam + r) * a.ld;
  // The row (L2-resident: the lm_head has just written it) is walked three times.  With one scalar load in flight per
  // thread the walks are bound by the L2 latency (32 warps x 128 B per ~700 cycles); each thread therefore takes groups
  // of four consecutive logits (one 16-byte load when the row is aligned) and requests four groups before it uses the
  // first.  A thread still meets its tokens in ascending index order, which the tie rule below relies on.
  const bool vec = (reinterpret_cast<uintptr_t>(row) & 15) == 0;
  const int nq = (V + 3) >> 2;
  auto load4 = [&](int q, float (&x)[4]) {
    if (q >= nq) {
      x[0] = x[1] = x[2] = x[3] = -INFINITY;
    } else if (vec && 4 * q + 3 < V) {
      const float4 t = *reinterpret_cast<const float4*>(row + 4 * q);
      x[0] = t.x; x[1] = t.y; x[2] = t.z; x[3] = t.w;
    } else {
#pragma unroll
      for (int e = 0; e < 4; ++e) x[e] = (4 * q + e < V) ? row[4 * q + e] : -INFINITY;
    }
  };
  const int qstep = blockDim.x;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
  // ---- walk 1: every thread's largest logit.  The beam-th largest of these thread maxima is a lower bound t0 of the
  // row's beam-th largest logit (they are `beam` different tokens), and hardly any token but those lies above it.
  float tmax = -INFINITY;
  for (int q0 = threadIdx.x; q0 < nq; q0 += 4 * qstep) {
    float x[4][4];
#pragma unroll
    for (int u = 0; u < 4; ++u) load4(q0 + u * qstep, x[u]);
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
      for (int e = 0; e < 4; ++e) tmax = fmaxf(tmax, x[u][e]);   // (-inf padding is neutral)
  }
  __shared__ float wtop[(kBeamRowThreads / 32) * kMaxBeam];
  __shared__ float s_t0, s_xmax;
  {
    float v = tmax;
    for (int k = 0; k < kMaxBeam; ++k) {   // the warp's k-th largest thread maximum
      float m = v;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
      if (lane == 0) wtop[w * kMaxBeam + k] = m;
      const unsigned holders = __ballot_sync(0xffffffffu, v == m);
      if (lane == __ffs(holders) - 1) v = -INFINITY;
    }
  }
  __syncthreads();
  if (w == 0) {
    float h[(kBeamRowThreads / 32) * kMaxBeam / 32];   // 4 values per lane
#pragma unroll
    for (int j = 0; j < (kBeamRowThreads / 32) * kMaxBeam / 32; ++j) {
      const int i = lane + 32 * j;
      h[j] = i < nw * kMaxBeam ? wtop[i] : -INFINITY;
    }
    float m = -INFINITY;
    for (int k = 0; k < beam; ++k) {
      float best = -INFINITY;
      int bj = 0;
#pragma unroll
      for (int j = 0; j < (kBeamRowThreads / 32) * kMaxBeam / 32; ++j)
        if (h[j] > best) { best = h[j]; bj = j; }
      m = best;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
      if (k == 0 && lane == 0) s_xmax = m;
      const unsigned holders = __ballot_sync(0xffffffffu, best == m);
      if (lane == __ffs(holders) - 1) {
#pragma unroll
        for (int j = 0; j < (kBeamRowThreads / 32) * kMaxBeam / 32; ++j)
          if (j == bj) h[j] = -INFINITY;
      }
    }
    if (lane == 0) s_t0 = m;
  }
  __shared__ int s_ncand;
  if (threadIdx.x == 0) s_ncand = 0;
  __syncthreads();
  const float xmax = s_xmax, t0 = s_t0;
  const float mx = unit_T ? xmax : xmax / T;     // == max of x / T: the division is monotone
  // The candidate value below is a non-decreasing function of the logit up to the rounding of expf / logf (< 1e-5 in the
  // log-probability, i.e. < 1e-5 T in the logit): every member of the row's top-beam has a logit above t0 minus that; the
  // margin taken is a hundred times wider.
  const float thr = t0 - (1e-3f * T + 1e-6f * fabsf(t0));
  constexpr int kCap = 128;
  __shared__ int cidx[kCap];
  __shared__ Cand cval[kCap];
  // ---- walk 2: softmax denominator; tokens above the threshold are noted
  float sm = 0.f;
  for (int q0 = threadIdx.x; q0 < nq; q0 += 4 * qstep) {
    float x[4][4];
#pragma unroll
    for (int u = 0; u < 4; ++u) load4(q0 + u * qstep, x[u]);
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        sm += expf((unit_T ? x[u][e] : x[u][e] / T) - mx);   // exp(-inf) == 0
        if (x[u][e] >= thr && x[u][e] != -INFINITY) {
          const int pos = atomicAdd(&s_ncand, 1);
          if (pos < kCap) cidx[pos] = 4 * (q0 + u * qstep) + e;
        }
      }
  }
  sm = block_sum(sm, fscratch);
  __syncthreads();
  const int ncand = s_ncand;
  if (ncand <= kCap) {
    // ---- the few candidates: exact values, then the best `beam` by (value, lowest flat index)
    if (threadIdx.x < kCap) {
      Cand c;
      c.v = -INFINITY;
      c.idx = 0x7fffffff;
      if (threadIdx.x < ncand) {
        const int v = cidx[threadIdx.x];
        const float x = row[v];
        const float lp = logf(expf((unit_T ? x : x / T) - mx) / sm);  // softmax(-1).log()
        c.v = first ? lp : (score + lp) / len;
        c.idx = r * V + v;
      }
      cval[threadIdx.x] = c;
    }
    __syncthreads();
    if (w == 0) {
      Cand mine[kCap / 32];
#pragma unroll
      for (int j = 0; j < kCap / 32; ++j) mine[j] = cval[lane + 32 * j];
      for (int k = 0; k < kMaxBeam; ++k) {
        Cand best;
        best.v = -INFINITY;
        best.idx = 0x7fffffff;
        int bj = -1;
        if (k < beam) {
#pragma unroll
          for (int j = 0; j < kCap / 32; ++j)
            if (mine[j].idx != 0x7fffffff && (bj < 0 || cand_better(mine[j], best))) { best = mine[j]; bj = j; }
        }
        Cand top = best;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          Cand oth;
          oth.v = __shfl_xor_sync(0xffffffffu, top.v, o);
          oth.idx = __shfl_xor_sync(0xffffffffu, top.idx, o);
          if (oth.idx != 0x7fffffff && (top.idx == 0x7fffffff || cand_better(oth, top))) top = oth;
        }
        if (bj >= 0 && top.idx == best.idx) {
#pragma unroll
          for (int j = 0; j < kCap / 32; ++j)
            if (j == bj) mine[j].idx = 0x7fffffff;
        }
        if (lane == 0) out[k] = top;
      }
    }
    return;
  }

  // ---- more than kCap tokens at the threshold (rows full of equal logits): per-thread lists over the whole row
  // thread-local top-kMaxBeam candidates (fixed size keeps them in registers; top-beam is a subset)
  Cand loc[kMaxBeam];
#pragma unroll
  for (int q = 0; q < kMaxBeam; ++q) {
    loc[q].v = -INFINITY;
    loc[q].idx = 0x7fffffff;
  }
  for (int v = threadIdx.x; v < V; v += blockDim.x) {   // (ascending index per thread: a later token never wins a tie)
    const float x = row[v];
    const float lp = logf(expf((unit_T ? x : x / T) - mx) / sm);  // softmax(-1).log()
    Cand c;
    c.v = first ? lp : (score + lp) / len;
    c.idx = r * V + v;
    if (!cand_better(c, loc[kMaxBeam - 1])) continue;
    loc[kMaxBeam - 1] = c;
#pragma unroll
    for (int q = kMaxBeam - 1; q > 0; --q) {
      if (cand_better(loc[q], loc[q - 1])) {
        const Cand t = loc[q];
        loc[q] = loc[q - 1];
        loc[q - 1] = t;
      }
    }
  }
  // warp merge: repeatedly extract the best head among the 32 lanes
  {
    int head = 0;
    for (int k = 0; k < beam; ++k) {
      Cand mine;
      mine.v = -INFINITY;
      mine.idx = 0x7fffffff;
#pragma unroll
      for (int q = 0; q < kMaxBeam; ++q)
        if (q == head) mine = loc[q];
      Cand best = mine;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        Cand oth;
        oth.v = __shfl_xor_sync(0xffffffffu, best.v, o);
        oth.idx = __shfl_xor_sync(0xffffffffu, best.idx, o);
        if (cand_better(oth, best)) best = oth;
      }
      if (best.idx == mine.idx && best.idx != 0x7fffffff) ++head;
      if (lane == 0) wcand[w * kMaxBeam + k] = best;
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    // final merge of the warps' sorted lists by one thread
    int heads[kBeamRowThreads / 32];
    for (int q = 0; q < nw; ++q) heads[q] = 0;
    for (int k = 0; k < kMaxBeam; ++k) {
      Cand best;
      best.v = -INFINITY;
      best.idx = 0x7fffffff;
      if (k < beam) {
        int bw = -1;
        for (int q = 0; q < nw; ++q) {
          if (heads[q] >= beam) continue;
          const Cand c = wcand[q * kMaxBeam + heads[q]];
          if (bw < 0 || cand_better(c, best)) {
            best = c;
            bw = q;
          }
        }
        heads[bw]++;
      }
      out[k] = best;
    }
  }
}

__global__ void __launch_bounds__(256) beam_merge_kernel(const BeamArgs a) {
  __shared__ Cand top[kMaxBeam];
  __shared__ float s_len[kMaxBeam];
  __shared__ uint8_t s_stop[kMaxBeam];
  extern __shared__ int perm_buf[];  // beam * max(max_len, max_pages) ints
  const int n = blockIdx.x;
  int g;
  if (beam_group(a, n, g)) return;
  const int beam = a.beam, V = a.V;
  const int step = a.grp.group_step ? a.grp.group_step[g] : *a.step;
  const bool first = (step == 0);
  const int rows = first ? 1 : beam;
  if (threadIdx.x < beam) {
    const uint8_t st = first ? 0 : a.has_stopped[g * beam + threadIdx.x];
    s_stop[threadIdx.x] = st;
    s_len[threadIdx.x] = first ? 1.f : a.seq_lengths[g * beam + threadIdx.x] + (st ? 0.f : 1.f);
  }
  if (threadIdx.x == 0) {
    // merge of the rows' sorted candidate lists
    const Cand* cand = a.cand + static_cast<long long>(n) * beam * kMaxBeam;
    int heads[kMaxBeam];
    for (int q = 0; q < kMaxBeam; ++q) heads[q] = 0;
    for (int k = 0; k < beam; ++k) {
      int bw = -1;
      Cand best;
      best.v = -INFINITY;
      best.idx = 0x7fffffff;
      for (int q = 0; q < rows; ++q) {
        if (heads[q] >= beam) continue;
        const Cand c = cand[q * kMaxBeam + heads[q]];
        if (bw < 0 || cand_better(c, best)) {
          best = c;
          bw = q;
        }
      }
      heads[bw]++;
      top[k] = best;
    }
  }
  __syncthreads();

  // bookkeeping
  __shared__ int s_src[kMaxBeam], s_tok[kMaxBeam];
  __shared__ float s_new_len[kMaxBeam], s_new_score[kMaxBeam];
  __shared__ uint8_t s_new_stop[kMaxBeam];
  if (threadIdx.x < beam) {
    const int k = threadIdx.x;
    const Cand c = top[k];
    int src, tok;
    float new_len, new_score;
    uint8_t stopped;
    if (first) {
      src = 0;
      tok = c.idx;
      new_len = 1.f;
      new_score = c.v;
      stopped = 0;
    } else {
      src = c.idx / V;
      tok = c.idx % V;
      new_len = s_len[src];
      new_score = c.v * new_len;
      stopped = s_stop[src];
    }
    stopped = stopped | (tok == a.stop_token ? 1 : 0);
    s_src[k] = src;
    s_tok[k] = tok;
    a.scores[g * beam + k] = new_score;
    a.seq_lengths[g * beam + k] = new_len;
    a.has_stopped[g * beam + k] = stopped;
    a.next_tokens[g * beam + k] = tok;
    a.src_rows[g * beam + k] = g * beam + src;
    s_new_stop[k] = stopped;
    s_new_len[k] = new_len;
    s_new_score[k] = new_score;
  }
  __syncthreads();
  // tokens = cat(tokens[src], tok)
  int* tk = a.tokens + static_cast<long long>(g) * beam * a.max_len;
  {
    if (!first) {
      for (int idx = threadIdx.x; idx < beam * step; idx += blockDim.x) perm_buf[idx] = tk[(idx / step) * a.max_len + idx % step];
      __syncthreads();
      for (int idx = threadIdx.x; idx < beam * step; idx += blockDim.x) {
        const int k = idx / step, t = idx % step;
        tk[k * a.max_len + t] = perm_buf[s_src[k] * step + t];
      }
    }
    if (threadIdx.x < beam && step < a.max_len) tk[threadIdx.x * a.max_len + step] = s_tok[threadIdx.x];
  }
  // block tables: row k inherits the cached-token entries of its source row
  // (in per-group mode including the token the decode step has just appended: ctx_len has not been advanced yet)
  int ctx = 0;
  if (!first && a.block_table != nullptr) {
    __syncthreads();
    ctx = a.ctx_len[g * beam] + (a.grp.group_step ? 1 : 0);
    int* bt = a.block_table + static_cast<long long>(g) * beam * a.max_pages;
    for (int idx = threadIdx.x; idx < beam * ctx; idx += blockDim.x) perm_buf[idx] = bt[(idx / ctx) * a.max_pages + idx % ctx];
    __syncthreads();
    for (int idx = threadIdx.x; idx < beam * ctx; idx += blockDim.x) {
      const int k = idx / ctx, t = idx % ctx;
      bt[k * a.max_pages + t] = perm_buf[s_src[k] * ctx + t];
    }
  }
  if (a.grp.group_step == nullptr) return;
  // per-group mode: advance the group; at its end (generate_beam's `if has_stopped.all(): break`, inference.py:70-148,
  // or max_len tokens) hand its beams to the caller's outputs
  __syncthreads();
  if (!first && threadIdx.x < beam) a.ctx_len[g * beam + threadIdx.x] = ctx;
  if (threadIdx.x == 0) a.grp.group_step[g] = step + 1;
  bool all_stopped = true;
  for (int k = 0; k < beam; ++k) all_stopped = all_stopped && s_new_stop[k];
  if (!all_stopped && step + 1 < a.max_len) return;
  const int img = a.grp.group_image[g];
  int* out_tokens = static_cast<int*>(a.grp.out[0]) + static_cast<long long>(img) * beam * a.max_len;
  for (int idx = threadIdx.x; idx < beam * a.max_len; idx += blockDim.x) out_tokens[idx] = tk[idx];
  if (threadIdx.x < beam) {
    static_cast<int*>(a.grp.out[1])[img * beam + threadIdx.x] = static_cast<int>(s_new_len[threadIdx.x]);
    static_cast<float*>(a.grp.out[2])[img * beam + threadIdx.x] = s_new_score[threadIdx.x] / s_new_len[threadIdx.x];
  }
  if (threadIdx.x == 0) a.grp.finished[g] = 1;
}

// ------------------------------------------------------------------------------------------------ bookkeeping
__global__ void advance_kernel(const int* __restrict__ next, int rows, int* tokens_out, int max_len, int* lengths,
                               int* stops, uint8_t* finished, int* ctx_len, int* step, int stop_token, int max_stops,
                               int eos_token) {
  ptx::grid_dep_wait();
  ptx::grid_dep_launch();
  const int st = *step;
  for (int r = threadIdx.x; r < rows; r += blockDim.x) {
    const int tok = next[r];
    if (tokens_out && st < max_len) tokens_out[static_cast<long long>(r) * max_len + st] = tok;
    if (finished && !finished[r]) {
      int sc = stops[r];
      if (tok == stop_token) sc += 1;
      stops[r] = sc;
      const bool fin = (max_stops > 0 && sc >= max_stops) || (eos_token >= 0 && tok == eos_token);
      lengths[r] = st + 1;
      if (fin) finished[r] = 1;
    }
    if (ctx_len) ctx_len[r] += 1;
  }
  __syncthreads();
  if (threadIdx.x == 0) *step = st + 1;
}

// the per-row mode (internal.h: RowAdvance)
__global__ void advance_rows_kernel(const int* __restrict__ next, int n, int* hist, int max_len, int* lengths, int* stops,
                                    uint8_t* finished, int* ctx_len, int stop_token, int max_stops, int eos_token,
                                    const RowAdvance ra) {
  ptx::grid_dep_wait();
  ptx::grid_dep_launch();
  int* out_tokens = static_cast<int*>(ra.out[0]);
  int* out_lengths = static_cast<int*>(ra.out[1]);
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const int r = ra.slots ? ra.slots[i] : i;
    const int img = ra.row_image[r];
    if (img < 0 || finished[r]) continue;
    const int tok = next[i];
    const int st = ra.row_step[r];
    hist[static_cast<long long>(r) * max_len + st] = tok;
    out_tokens[static_cast<long long>(img) * max_len + st] = tok;
    out_lengths[img] = st + 1;
    const int sc = stops[r] + (tok == stop_token ? 1 : 0);
    stops[r] = sc;
    lengths[r] = st + 1;
    if ((max_stops > 0 && sc >= max_stops) || (eos_token >= 0 && tok == eos_token) || st + 1 >= max_len) finished[r] = 1;
    if (ctx_len) ctx_len[r] += 1;
    ra.row_step[r] = st + 1;
    if (ra.next_tokens) ra.next_tokens[r] = tok;
  }
}

}  // namespace

int sample_greedy(const float* logits, long long ld, int B, int V, int* next, cudaStream_t s) {
  if (B <= 0) return 0;
  cudaError_t e = launch_kernel(greedy_kernel, dim3(B), dim3(kSampThreads), 0, s, true, logits, ld, V, next);
  return e == cudaSuccess ? 0 : (int)e;
}

int cross_entropy(const float* logits, long long ld, int rows, int V, const int* targets, const int* row_map, int ignore_index,
                  float* row_loss, float* out2, cudaStream_t s) {
  if (rows <= 0) return 0;
  cross_entropy_rows_kernel<<<rows, kSampThreads, 0, s>>>(logits, ld, V, targets, row_map, ignore_index, row_loss);
  cross_entropy_mean_kernel<<<1, kSampThreads, 0, s>>>(row_loss, targets, rows, ignore_index, out2);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? 0 : (int)e;
}

int sample_top_p(const float* logits, long long ld, int B, int V, const SampleParams& sp, int* next,
                 cudaStream_t s) {
  if (B <= 0) return 0;
  const size_t smem = static_cast<size_t>(V) * sizeof(float);
  if (smem > 208 * 1024) return (int)cudaErrorInvalidValue;
  static bool configured_dev[kMaxDevices] = {};
  bool& configured = configured_dev[current_device_slot()];
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(top_p_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 208 * 1024);
    if (e != cudaSuccess) return (int)e;
    configured = true;
  }
  TopPArgs a;
  a.logits = logits; a.ld = ld; a.V = V;
  a.temperature = sp.temperature; a.top_p = sp.top_p; a.top_k = sp.top_k;
  a.top_p_rows = sp.top_p_rows; a.top_k_rows = sp.top_k_rows;
  a.typ_p = sp.typ_p; a.typ_p_rows = sp.typ_p_rows;
  a.rep_pen = sp.repetition_penalty; a.history = sp.history; a.ld_hist = sp.ld_hist;
  a.hist_len = sp.hist_len; a.hist_len_scalar = sp.hist_len_scalar; a.hist_len_from_step = sp.hist_len_from_step;
  a.q_noise = sp.q_noise; a.ldq = sp.ldq; a.q_step_stride = sp.q_step_stride; a.seed = sp.seed; a.row_ids = sp.row_ids;
  a.step = sp.step; a.step_scalar = sp.step_scalar; a.row_step = sp.row_step;
  a.filtered_out = sp.filtered_out; a.alt_out = sp.alt_out; a.next = next;
  static const bool fast_on = [] {   // CCB_SAMPLER_FAST=0: always the radix select (A/B)
    const char* e = getenv("CCB_SAMPLER_FAST");
    return !(e && e[0] == '0');
  }();
  a.fast = fast_on ? 1 : 0;
  top_p_kernel<<<B, kSampThreads, smem, s>>>(a);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? 0 : (int)e;
}

int beam_step(const float* logits, long long ld, int N, int beam, int V, float temperature, int stop_token,
              const BeamState& st, int* next_tokens, int* src_rows, int* block_table, int max_pages,
              int* ctx_len, cudaStream_t s, const BeamGroups* groups) {
  if (N <= 0) return 0;
  if (beam < 1 || beam > kMaxBeam) return (int)cudaErrorInvalidValue;
  BeamArgs a;
  a.logits = logits; a.ld = ld; a.beam = beam; a.V = V; a.temperature = temperature; a.stop_token = stop_token;
  a.scores = st.scores; a.seq_lengths = st.seq_lengths; a.has_stopped = st.has_stopped; a.tokens = st.tokens;
  a.max_len = st.max_len; a.step = st.step; a.next_tokens = next_tokens; a.src_rows = src_rows;
  a.block_table = block_table; a.max_pages = max_pages; a.ctx_len = ctx_len;
  if (groups) {
    if (!groups->group_step || !groups->group_image || !groups->finished || !groups->out || !block_table || !ctx_len)
      return (int)cudaErrorInvalidValue;
    a.grp = *groups;
  }
  if (st.cand_scratch == nullptr || st.cand_rows < N * beam) return (int)cudaErrorInvalidValue;
  a.cand = static_cast<Cand*>(st.cand_scratch);
  const size_t smem = beam_merge_smem(beam, st.max_len, max_pages);
  if (smem > kBeamMergeMaxSmem) return (int)cudaErrorInvalidValue;
  static bool configured_dev[kMaxDevices] = {};
  bool& configured = configured_dev[current_device_slot()];
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(beam_merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(kBeamMergeMaxSmem));
    if (e != cudaSuccess) return (int)e;
    configured = true;
  }
  beam_rows_kernel<<<N * beam, kBeamRowThreads, 0, s>>>(a);
  beam_merge_kernel<<<N, 256, smem, s>>>(a);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? 0 : (int)e;
}

__global__ void increment_kernel(int* x, int rows, int* scalar) {
  for (int r = threadIdx.x; r < rows; r += blockDim.x) x[r] += 1;
  if (scalar && threadIdx.x == 0) *scalar += 1;
}
}  // namespace ccb
namespace ccb {
int increment_rows(int* x, int rows, int* scalar, cudaStream_t s) {
  increment_kernel<<<1, 1024, 0, s>>>(x, rows, scalar);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? 0 : (int)e;
}

int advance_rows(const int* next, int rows, int* tokens_out, int max_len, int* lengths, int* stops, uint8_t* finished,
                 int* ctx_len, int* step, int stop_token, int max_stops, int eos_token, cudaStream_t s,
                 const RowAdvance* per_row) {
  if (per_row) {
    if (!per_row->row_step || !per_row->row_image || !per_row->out || !tokens_out || !lengths || !stops || !finished)
      return (int)cudaErrorInvalidValue;
    const cudaError_t e = launch_kernel(advance_rows_kernel, dim3(1), dim3(1024), 0, s, true, next, rows, tokens_out, max_len,
                                        lengths, stops, finished, ctx_len, stop_token, max_stops, eos_token, *per_row);
    return e == cudaSuccess ? 0 : (int)e;
  }
  cudaError_t e = launch_kernel(advance_kernel, dim3(1), dim3(1024), 0, s, true, next, rows, tokens_out, max_len, lengths,
                                stops, finished, ctx_len, step, stop_token, max_stops, eos_token);
  return e == cudaSuccess ? 0 : (int)e;
}

}  // namespace ccb
