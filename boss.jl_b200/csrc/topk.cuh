// topk.cuh -- the k best candidates of a scoring call, kept on the device (boss_ei_score_topk, DESIGN.md 2.10).
//
//   select_*_kernel   keep the `target` best of (running set, new values): radix select of the target-th key over
//                     8 passes of 8 bits, then an ordered compaction (everything above that key, then the lowest
//                     positions among the keys equal to it)
//   topk_sort_kernel  the final <= TOPK_MAX survivors, bitonic-sorted by (key descending, position ascending) in one CTA
//
// Order: Julia's isless, descending, ties to the lower index (stable sortperm(vals; rev=true)); the running set and
// every new batch are in ascending index order, so position order is index order throughout.  Counts are the only
// atomics, so the result does not depend on scheduling, chunk size or how candidates are split across devices.
#pragma once
#include "score.cuh"

namespace boss {

constexpr int TOPK_MAX = 8192;                              // largest k of a top-k call
constexpr int TOPK_SORT_SMEM = TOPK_MAX * (8 + 4);          // 96 KB: keys + positions of the final sort

// isless order as unsigned 64-bit keys: NaN the top key (all NaNs equal), -0.0 below +0.0
__device__ __forceinline__ unsigned long long isless_key(double v) {
  if (v != v) return ~0ull;
  const unsigned long long u = (unsigned long long)__double_as_longlong(v);
  return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}

// the elements of one selection: positions [0, r) are the running set, [r, r + n) the new values (index idx0 + i)
struct SelectIn {
  const double *run_val;
  const long long *run_idx;
  int r;
  const double *val;
  long long idx0;
  int n;
  int nan_low;   // 1: NaN lowest (bound_key, the seed of a screened call), 0: isless order
  __device__ __forceinline__ double value(int i) const { return i < r ? run_val[i] : val[i - r]; }
  __device__ __forceinline__ long long index(int i) const { return i < r ? run_idx[i] : idx0 + (i - r); }
  __device__ __forceinline__ unsigned long long key(int i) const {
    const double v = value(i);
    return nan_low ? bound_key(v) : isless_key(v);
  }
};

// the target-th key as it is being found: its high bits (prefix), and how many of the elements matching the prefix
// still have to be taken
struct SelectState {
  unsigned long long prefix;
  int need;
  unsigned int hist[256];
};

// one CTA of 256.  With need = every element and no histogram pass, prefix 0 keeps them all (every key is >= 0).
__global__ void select_init_kernel(SelectState *st, int need) {
  if (threadIdx.x == 0) {
    st->prefix = 0ull;
    st->need = need;
  }
  st->hist[threadIdx.x] = 0u;
}

// histogram of bits [shift, shift + 8) over the elements whose higher bits equal the prefix
__global__ void __launch_bounds__(256) select_hist_kernel(SelectIn in, SelectState *st, int shift) {
  __shared__ unsigned int h[256];
  h[threadIdx.x] = 0u;
  __syncthreads();
  const unsigned long long hi = shift >= 56 ? 0ull : (~0ull << (shift + 8));
  const unsigned long long pre = st->prefix & hi;
  const int N = in.r + in.n;
  for (int i = blockIdx.x * 256 + threadIdx.x; i < N; i += gridDim.x * 256) {
    const unsigned long long k = in.key(i);
    if ((k & hi) == pre) atomicAdd(&h[(k >> shift) & 255], 1u);
  }
  __syncthreads();
  if (h[threadIdx.x]) atomicAdd(&st->hist[threadIdx.x], h[threadIdx.x]);
}

// the digit of the target-th key: the highest bin whose count, with the bins above it, reaches `need`
__global__ void __launch_bounds__(256) select_scan_kernel(SelectState *st, int shift) {
  __shared__ unsigned int h[256];
  h[threadIdx.x] = st->hist[threadIdx.x];
  st->hist[threadIdx.x] = 0u;
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned int need = (unsigned int)st->need;
    unsigned int above = 0u;
    int b = 255;
    for (; b > 0; --b) {
      if (above + h[b] >= need) break;
      above += h[b];
    }
    st->prefix |= (unsigned long long)b << shift;
    st->need = (int)(need - above);
  }
}

// per 256 positions: keys above the target-th key, keys equal to it
__global__ void __launch_bounds__(256) select_count_kernel(SelectIn in, const SelectState *st, int2 *cnt) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  const unsigned long long K = st->prefix;
  const bool ok = i < in.r + in.n;
  const unsigned long long k = ok ? in.key(i) : 0ull;
  const int g = __syncthreads_count(ok && k > K);
  const int e = __syncthreads_count(ok && k == K);
  if (threadIdx.x == 0) cnt[blockIdx.x] = make_int2(g, e);
}

// ordered compaction: keys above K, then the first `need` keys equal to K, in position order
__global__ void __launch_bounds__(256) select_compact_kernel(SelectIn in, const SelectState *st, const int2 *cnt,
                                                             double *out_val, long long *out_idx) {
  __shared__ int s_gt, s_eq;
  __shared__ int w_gt[8], w_eq[8];
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, b = blockIdx.x;
  if (w == 0) {
    int g = 0, e = 0;
    for (int j = lane; j < b; j += 32) {
      const int2 c = cnt[j];
      g += c.x;
      e += c.y;
    }
    for (int o = 16; o > 0; o >>= 1) {
      g += __shfl_xor_sync(0xffffffffu, g, o);
      e += __shfl_xor_sync(0xffffffffu, e, o);
    }
    if (lane == 0) {
      s_gt = g;
      s_eq = e;
    }
  }
  const int i = b * 256 + tid;
  const unsigned long long K = st->prefix;
  const int need = st->need;
  const bool ok = i < in.r + in.n;
  const unsigned long long k = ok ? in.key(i) : 0ull;
  const bool gt = ok && k > K, eq = ok && k == K;
  const unsigned bg = __ballot_sync(0xffffffffu, gt), be = __ballot_sync(0xffffffffu, eq);
  if (lane == 0) {
    w_gt[w] = __popc(bg);
    w_eq[w] = __popc(be);
  }
  __syncthreads();
  if (!gt && !eq) return;
  const unsigned below = (1u << lane) - 1u;
  int g_before = s_gt + __popc(bg & below), e_before = s_eq + __popc(be & below);
  for (int q = 0; q < w; ++q) {
    g_before += w_gt[q];
    e_before += w_eq[q];
  }
  if (eq && e_before >= need) return;
  const int pos = g_before + min(e_before, need);
  out_val[pos] = in.value(i);
  out_idx[pos] = in.index(i);
}

// One CTA: the r survivors (positions in ascending index order) sorted by (isless key descending, position
// ascending); row e of the result is value val[pos], index map ? map[idx[pos]] : idx[pos].  P = power of two >= r.
__global__ void __launch_bounds__(1024) topk_sort_kernel(const double *val, const long long *idx, int r, int P,
                                                         const long long *map, double *out_val, long long *out_idx) {
  extern __shared__ unsigned long long topk_sm[];
  unsigned long long *sk = topk_sm;
  int *sp = reinterpret_cast<int *>(topk_sm + P);
  const int tid = threadIdx.x;
  for (int e = tid; e < P; e += 1024) {
    sk[e] = e < r ? isless_key(val[e]) : 0ull;   // padding: below every real key (NaN-free keys are > 0), last position
    sp[e] = e < r ? e : 0x7fffffff;
  }
  for (int k = 2; k <= P; k <<= 1)
    for (int j = k >> 1; j > 0; j >>= 1) {
      __syncthreads();
      for (int t = tid; t < (P >> 1); t += 1024) {
        const int a = ((t & ~(j - 1)) << 1) | (t & (j - 1)), b = a | j;
        const bool b_first = sk[b] > sk[a] || (sk[b] == sk[a] && sp[b] < sp[a]);
        if (b_first == ((a & k) == 0)) {
          const unsigned long long tk = sk[a];
          sk[a] = sk[b];
          sk[b] = tk;
          const int tp = sp[a];
          sp[a] = sp[b];
          sp[b] = tp;
        }
      }
    }
  __syncthreads();
  for (int e = tid; e < r; e += 1024) {
    const int p = sp[e];
    const long long ix = idx[p];
    out_val[e] = val[p];
    out_idx[e] = map ? map[ix] : ix;
  }
}

}  // namespace boss
