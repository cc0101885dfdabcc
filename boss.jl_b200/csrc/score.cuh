// score.cuh -- the acquisition-scoring path (SURVEY.md 8 rows a3-a7) for one chunk of candidates:
//
//   xcov_kernel        K*^T tile-packed (cand x train) + mu = K*^T alpha        [FP64 pipe: exp/sqrt]
//   score_trmm_kernel  q_m = | W k*_m |^2, V = W K* never leaves the SM          [DMMA, TMA-fed]
//   acq_kernel         var = a^2 - q + 1e-18, _clip_var, EI x PoF, guards, per-block argmax  [HBM]
//   argmax_final_kernel  deterministic reduction of the block winners
//
// Reference: mean_and_var(::GaussianProcessPosterior, X) src/models/gaussian_process.jl:174-178 ->
// AbstractGPs mean_and_var(PosteriorGP) (k* , U'\k*, colsum of squares); expected_improvement.jl:58-114;
// argmax loops grid.jl:52-65, sampling.jl:37-48.  W = L^-1 is formed once per fit, so the per-candidate
// triangular solve of the reference becomes a triangular matrix product.
#pragma once
#include "acq.cuh"
#include "gemm_core.cuh"
#include "kernel_fn.cuh"
#include "tk_params.cuh"

namespace boss {

// ---------------------------------------------------------------------------------------------
// cross-covariance of a candidate chunk with the training set, + posterior mean
// ---------------------------------------------------------------------------------------------


// grid = (candidate blocks, splits over the 128-point training chunks).  Every chunk's contribution to
// mu is written as its own partial (fixed summation order downstream), so results do not depend on the split.

// sum_{q = 0}^{P-1} base[q * stride] added in ascending q (the fixed order that makes results split-invariant), with the
// loads issued 16 at a time: these reductions run on a handful of threads in the small-batch paths, where a chain of
// P dependent load -> add steps costs P memory latencies (8-12 us per launch at n = 4096)
__device__ __forceinline__ double ordered_sum(const double *__restrict__ base, size_t stride, int P) {
  double acc = 0.0;
  int q = 0;
  for (; q + 16 <= P; q += 16) {
    double v[16];
#pragma unroll
    for (int u = 0; u < 16; ++u) v[u] = base[(size_t)(q + u) * stride];
#pragma unroll
    for (int u = 0; u < 16; ++u) acc += v[u];
  }
  for (; q < P; ++q) acc += base[(size_t)q * stride];
  return acc;
}

// out[c] = sum_{p = 0}^{P-1} in[p*ld + c]  (ascending p)
__global__ void __launch_bounds__(256) reduce_rows_kernel(const double *__restrict__ in, int P, size_t ld,
                                                          double *__restrict__ out, int count) {
  const int c = blockIdx.x * 256 + threadIdx.x;
  if (c >= count) return;
  out[c] = ordered_sum(in + c, ld, P);
}

// ---------------------------------------------------------------------------------------------
// elementwise acquisition stage + block argmax
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) acq_kernel(AcqParams p) {
  __shared__ double sv[256];
  __shared__ long long si[256];
  const int tid = threadIdx.x;
  const int c = blockIdx.x * 256 + tid;
  const long long m = p.m0 + c;
  const bool active = (c < p.chunk) && (m < p.M);
  const double result = active ? acq_candidate(p, c, m) : -INFINITY;
  if (p.blk_val == nullptr) return;
  // block argmax with Julia semantics (first maximal, NaN maximal); inactive lanes carry idx = LLONG_MAX
  sv[tid] = result;
  si[tid] = active ? m : 0x7fffffffffffffffLL;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (tid < o) {
      const double v2 = sv[tid + o];
      const long long i2 = si[tid + o];
      const bool a1 = si[tid] != 0x7fffffffffffffffLL, a2 = i2 != 0x7fffffffffffffffLL;
      if (a2 && (!a1 || acq_better(v2, i2, sv[tid], si[tid]))) {
        sv[tid] = v2;
        si[tid] = i2;
      }
    }
    __syncthreads();
  }
  if (tid == 0) {
    p.blk_val[blockIdx.x] = sv[0];
    p.blk_idx[blockIdx.x] = si[0];
  }
}

// Fold `nblk` block winners into the running (val, idx) pair held in best[0], bidx[0].
__global__ void argmax_final_kernel(const double *blk_val, const long long *blk_idx, int nblk, double *best,
                                    long long *bidx) {
  __shared__ double sv[256];
  __shared__ long long si[256];
  const int tid = threadIdx.x;
  double v = 0.0;
  long long ix = 0x7fffffffffffffffLL;
  for (int b = tid; b < nblk; b += 256) {
    const long long i2 = blk_idx[b];
    if (i2 != 0x7fffffffffffffffLL && (ix == 0x7fffffffffffffffLL || acq_better(blk_val[b], i2, v, ix))) {
      v = blk_val[b];
      ix = i2;
    }
  }
  sv[tid] = v;
  si[tid] = ix;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (tid < o) {
      const long long i2 = si[tid + o];
      if (i2 != 0x7fffffffffffffffLL && (si[tid] == 0x7fffffffffffffffLL || acq_better(sv[tid + o], i2, sv[tid], si[tid]))) {
        sv[tid] = sv[tid + o];
        si[tid] = i2;
      }
    }
    __syncthreads();
  }
  if (tid == 0 && si[0] != 0x7fffffffffffffffLL) {
    if (*bidx < 0 || acq_better(sv[0], si[0], *best, *bidx)) {
      *best = sv[0];
      *bidx = si[0];
    }
  }
}

// ---------------------------------------------------------------------------------------------
// argmax screening (DESIGN.md 2.9).  acq_kernel with sumsq == null and PoF / guards off writes, per candidate, the
// EI at the prior standard deviation: an upper bound of its acquisition.  A candidate whose bound is below the exact
// score of some candidate (the best of a small seed batch) cannot be the argmax; the others are compacted, in
// ascending order, into a pool that the ordinary chunk loop scores.
// ---------------------------------------------------------------------------------------------
constexpr int SEED_N = 128;     // seed candidates: the highest bounds of the first chunk
constexpr int TOPK_IN = 2048;   // elements one CTA of seed_topk_kernel sorts

// larger bound -> larger key; NaN lowest (a NaN bound is kept by the compaction anyway, it is not worth a seed slot)
__device__ __forceinline__ unsigned long long bound_key(double b) {
  if (b != b) return 0ull;
  const unsigned long long u = (unsigned long long)__double_as_longlong(b);
  return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}

// The SEED_N best of each TOPK_IN inputs (key descending, then index ascending) in that order; the inputs are the
// bounds of a chunk (bounds != null, index = position) or the (key, index) output of an earlier round.
__global__ void __launch_bounds__(1024) seed_topk_kernel(const double *bounds, const unsigned long long *kin,
                                                         const int *iin, int n, unsigned long long *kout, int *iout) {
  __shared__ unsigned long long sk[TOPK_IN];
  __shared__ int si[TOPK_IN];
  const int tid = threadIdx.x, base = blockIdx.x * TOPK_IN;
  for (int e = tid; e < TOPK_IN; e += 1024) {
    const int g = base + e;
    unsigned long long k = 0ull;
    int i = 0x7fffffff;   // padding sorts last
    if (g < n) {
      k = bounds ? bound_key(bounds[g]) : kin[g];
      i = bounds ? g : iin[g];
    }
    sk[e] = k;
    si[e] = i;
  }
  for (int k = 2; k <= TOPK_IN; k <<= 1)   // bitonic sort, one compare-exchange per thread and step
    for (int j = k >> 1; j > 0; j >>= 1) {
      __syncthreads();
      const int a = ((tid & ~(j - 1)) << 1) | (tid & (j - 1)), b = a | j;
      const bool b_first = sk[b] > sk[a] || (sk[b] == sk[a] && si[b] < si[a]);
      if (b_first == ((a & k) == 0)) {
        const unsigned long long tk = sk[a];
        sk[a] = sk[b];
        sk[b] = tk;
        const int ti = si[a];
        si[a] = si[b];
        si[b] = ti;
      }
    }
  __syncthreads();
  if (tid < SEED_N) {
    kout[blockIdx.x * SEED_N + tid] = sk[tid];
    iout[blockIdx.x * SEED_N + tid] = si[tid];
  }
}

// row s of the seed batch = candidate sel[s] of the chunk (xs / pm / cm point at the chunk's first candidate)
template <typename I>
__global__ void seed_gather_kernel(const I *sel, int ns, const double *xs, const double *pm, const unsigned char *cm,
                                   int d, int y_dim, double *sx, double *spm, unsigned char *scm) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= ns) return;
  const size_t c = (size_t)sel[s];
  for (int j = 0; j < d; ++j) sx[(size_t)s * d + j] = xs[c * d + j];
  if (pm)
    for (int i = 0; i < y_dim; ++i) spm[(size_t)s * y_dim + i] = pm[c * y_dim + i];
  if (cm) scm[s] = cm[c];
}

// a candidate stays unless its bound is below thr = T (1 - 2^-30); a NaN bound stays.  With a verdict array (the
// re-compaction of the pool), rows whose verdict is not 1 (dropped by the FP64 refinement) go too.
__device__ __forceinline__ bool screen_keep(const double *bound, const unsigned char *ver, int c, int ch, double thr) {
  return c < ch && !(bound[c] < thr) && (!ver || ver[c] == 1);
}

// survivors per 128 candidates (launched with 128 threads)
__global__ void __launch_bounds__(128) screen_count_kernel(const double *bound, const unsigned char *ver, int ch, double thr,
                                                           long long *cnt) {
  const int k = __syncthreads_count(screen_keep(bound, ver, blockIdx.x * 128 + threadIdx.x, ch, thr));
  if (threadIdx.x == 0) cnt[blockIdx.x] = k;
}

// The n per-128 survivor counts become, in place, the pool offsets of their candidate blocks: base[par] plus the
// exclusive prefix sum.  base[par ^ 1] gets the pool size after them.  One CTA; each thread takes a contiguous run.
__global__ void __launch_bounds__(1024) screen_scan_kernel(long long *cnt, int n, long long *base, int par) {
  __shared__ long long ws[32];
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, per = (n + 1023) / 1024;
  const int j0 = min(n, tid * per), j1 = min(n, j0 + per);
  long long s = 0;
  for (int j = j0; j < j1; ++j) s += cnt[j];
  long long v = s;   // inclusive scan: within the warp, then over the warps
  for (int o = 1; o < 32; o <<= 1) {
    const long long u = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v += u;
  }
  if (lane == 31) ws[w] = v;
  __syncthreads();
  if (w == 0) {
    long long x = ws[lane];
    for (int o = 1; o < 32; o <<= 1) {
      const long long u = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x += u;
    }
    ws[lane] = x;
  }
  __syncthreads();
  long long off = base[par] + (w ? ws[w - 1] : 0) + v - s;
  for (int j = j0; j < j1; ++j) {
    const long long k = cnt[j];
    cnt[j] = off;
    off += k;
  }
  if (tid == 1023) base[par ^ 1] = off;
}

// ---- the FP32 mean tier (DESIGN.md 2.9) ----

// Per call and slice (one CTA of 1024 threads, every sum in a fixed order): the centre c = the mean of the n scaled
// training inputs; the FP32 copies the MMA tier reads (ScreenSlice: the TF32-split B fragments of t~ = fp32(ut - c),
// |t~|^2 and alpha); and the constants of the error bound, A1 = sum_j |alpha_j| and A3 = sum_j |alpha_j| |ut_j - c|^2.
// A = [A1, A3, c_0 .. c_{DP-1}].
__global__ void __launch_bounds__(1024) screen_consts_kernel(const double *Xt, const double *alpha, int n, int n_pad,
                                                             int DP, float *tfrag, float *tn_al, double *A) {
  __shared__ double s1[1024], s2[1024];
  __shared__ double wsum[32][32], cen[32];
  const int tid = threadIdx.x, KS = (DP + 7) / 8;
  for (int i = 0; i < DP; ++i) {   // per dimension: strided per-thread sums, a warp butterfly, the 32 warps in order
    double s = 0.0;
    for (int j = tid; j < n; j += 1024) s += Xt[(size_t)j * DP + i];
    for (int o = 1; o < 32; o <<= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((tid & 31) == 0) wsum[tid >> 5][i] = s;
  }
  __syncthreads();
  if (tid < DP) {
    double s = 0.0;
    for (int k = 0; k < 32; ++k) s += wsum[k][tid];
    cen[tid] = s / n;
    A[2 + tid] = cen[tid];
  }
  __syncthreads();
  double a1 = 0.0, a2 = 0.0;
  for (int j = tid; j < n_pad; j += 1024) {
    const double aj = fabs(alpha[j]);
    double n2 = 0.0;
    for (int i = 0; i < 8 * KS; ++i) {
      const double v = i < DP ? Xt[(size_t)j * DP + i] - cen[i] : 0.0;
      n2 = fma(v, v, n2);
      float hi, lo;
      tf32_split((float)v, hi, lo);
      // tile j / 8, k-step i / 8, lane 4 (j % 8) + i % 4; b0 holds dimension i % 8 < 4, b1 the others
      const size_t f = (((size_t)(j >> 3) * KS + (i >> 3)) * 32 + 4 * (j & 7) + (i & 3)) * 4 + ((i >> 2) & 1);
      tfrag[f] = hi;
      tfrag[f + 2] = lo;
    }
    tn_al[4 * (j >> 1) + (j & 1)] = (float)n2;   // the norms and the alphas of points 2i, 2i + 1 as FP32 pairs
    tn_al[4 * (j >> 1) + 2 + (j & 1)] = (float)alpha[j];
    a1 += aj;
    a2 = fma(aj, n2, a2);
  }
  s1[tid] = a1;
  s2[tid] = a2;
  __syncthreads();
  for (int o = 512; o > 0; o >>= 1) {
    if (tid < o) {
      s1[tid] += s1[tid + o];
      s2[tid] += s2[tid + o];
    }
    __syncthreads();
  }
  if (tid == 0) {
    A[0] = s1[0];
    A[1] = s2[0];
  }
}

// The ambiguous rows (verdict 2) among pool rows [0, n) of a piece: their candidates, prior means and rows, in any order
// (each gets its own verdict back); the count goes to cnt[0].
__global__ void __launch_bounds__(256) screen_amb_gather_kernel(const unsigned char *ver, int n, const double *px,
                                                                const double *ppm, int d, int y_dim, int r0, double *rx,
                                                                double *rpm, int *rrow, int *cnt) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i >= n || ver[i] != 2) return;
  const int s = atomicAdd(cnt, 1);
  for (int j = 0; j < d; ++j) rx[(size_t)s * d + j] = px[(size_t)i * d + j];
  if (ppm)
    for (int k = 0; k < y_dim; ++k) rpm[(size_t)s * y_dim + k] = ppm[(size_t)i * y_dim + k];
  rrow[s] = r0 + i;
}

// today's rule on the FP64 bounds of the gathered rows: verdict 1 (keep) unless bound < thr; the bound goes with it
__global__ void __launch_bounds__(256) screen_amb_scatter_kernel(const double *b, const int *rrow, int n, double thr,
                                                                 double *pbound, unsigned char *pver) {
  const int s = blockIdx.x * 256 + threadIdx.x;
  if (s >= n) return;
  const int row = rrow[s];
  pbound[row] = b[s];
  pver[row] = !(b[s] < thr) ? 1 : 0;
}

// the bounds the re-seed selects from: dropped rows count as NaN (lowest)
__global__ void __launch_bounds__(256) screen_sel_bound_kernel(const double *pbound, const unsigned char *pver, int n,
                                                               double *out) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i < n) out[i] = pver[i] == 1 ? pbound[i] : NAN;
}

struct CompactParams {
  const double *bound;
  const unsigned char *ver;      // re-compaction: the rows' verdicts (keep only 1), else null
  int ch;
  double thr;
  const double *lo;              // FP32 tier: EI at mu~ - E' (survivors with lo >= thr_keep are definite keeps), else null
  double thr_keep;
  const long long *off;          // pool offset of each 128 candidates (screen_scan_kernel)
  long long m0;                  // index (within the call) of the chunk's first candidate
  const double *xs, *pm;         // the chunk's first candidate (pm may be null)
  const unsigned char *cm;       // or null
  int d, y_dim;
  double *px, *ppm;              // pool: candidates, prior means,
  unsigned char *pcm;            //       constraint-mask entries,
  long long *pidx;               //       index within the call (m0 + position, or sidx[position] if sidx is set)
  const long long *sidx;
  double *pbound;                //       bounds (or null): hi in the FP32 tier, the FP64 bound otherwise
  unsigned char *pver;           //       verdicts (or null): 1 keep, 2 ambiguous (refined in Screen::finish)
};

// ordered compaction, 128 candidates per CTA: survivors keep their relative order, so the pool's first-maximal argmax
// is the call's
__global__ void __launch_bounds__(128) screen_compact_kernel(CompactParams p) {
  __shared__ int s_warp[4];
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, c = blockIdx.x * 128 + tid;
  const bool keep = screen_keep(p.bound, p.ver, c, p.ch, p.thr);
  const unsigned bal = __ballot_sync(0xffffffffu, keep);
  if (lane == 0) s_warp[w] = __popc(bal);
  __syncthreads();
  if (!keep) return;
  long long o = p.off[blockIdx.x] + __popc(bal & ((1u << lane) - 1u));
  for (int q = 0; q < w; ++q) o += s_warp[q];
  for (int j = 0; j < p.d; ++j) p.px[o * p.d + j] = p.xs[(size_t)c * p.d + j];
  if (p.pm)
    for (int i = 0; i < p.y_dim; ++i) p.ppm[o * p.y_dim + i] = p.pm[(size_t)c * p.y_dim + i];
  if (p.cm) p.pcm[o] = p.cm[c];
  p.pidx[o] = p.sidx ? p.sidx[c] : p.m0 + c;
  if (p.pbound) p.pbound[o] = p.bound[c];
  if (p.pver) p.pver[o] = (!p.lo || p.lo[c] >= p.thr_keep) ? 1 : 2;
}

// ---------------------------------------------------------------------------------------------
// fused triangular product + column sum of squares:  q[m] = sum_r ( sum_{k<=r} W[r][k] K*[k][m] )^2
// One CTA owns 128 candidates and walks all row blocks of W; the ring streams W (L2-resident) and the
// CTA's K*^T block (re-read once per row block, triangular k-range).
// ---------------------------------------------------------------------------------------------
struct ScoreParams {
  const double *W;    // P-layout n_pad x n_pad lower-triangular inverse factor
  const double *Ks;   // chunk scratch
  int nblk, ktiles;
  double *ss_part;    // [2*nblk][ld] per-(row block, warp-row half) partial sums of squares
  int ld;
  double *VT;         // optional chunk scratch (P-layout, rows = candidates): V = W K* stored transposed (gradient mode)
  // fused epilogue (one CTA walks ALL row blocks of its candidate block, last slice of the chunk): the column sums
  // of squares stay in registers, and the CTA finishes its 128 candidates itself -- mean, variance, EI x PoF, guards,
  // block argmax -- and the last CTA of the launch folds the block winners into the running (value, index) pair.
  int fused;
  AcqParams ap;             // ap.mu / ap.sumsq rows of the other slices were written by earlier launches
  const double *mu_part;    // xcov's partials for this slice, [P][ld]
  int P;
  double *mu_row, *ss_row;  // this slice's rows of ap.mu / ap.sumsq
  double *best;             // running winner of the call (device)
  long long *bidx;
  unsigned int *counter;    // CTAs of this launch that have finished (reset by the last one)
};

// Row blocks of a triangular operand are dealt to the `ns` CTAs of a candidate block in zig-zag order
// (split y gets y, 2ns-1-y, 2ns+y, 4ns-1-y, ...), which balances the triangular work; ns = 1 is the plain walk.
__device__ __forceinline__ int zigzag_row(int j, int y, int ns2) { return (j >> 1) * ns2 + ((j & 1) ? ns2 - 1 - y : y); }

struct ScoreIt {
  const double *w;       // W (lower triangular): row block i uses k-tiles 0 .. 8(i+1)-1
  const double *ks;      // first tile of this CTA's K*^T block
  int j, i, kt, nblk, ktiles, y, ns2;
  __device__ __forceinline__ bool valid() const { return i < nblk; }
  __device__ __forceinline__ const double *A() const { return w + ((size_t)i * ktiles + kt) * TILE_ELEMS; }
  __device__ __forceinline__ const double *B() const { return ks + (size_t)kt * TILE_ELEMS; }
  __device__ __forceinline__ bool tile_end() const { return kt == (i + 1) * KT_PER_BLOCK - 1; }
  __device__ __forceinline__ int tile() const { return i; }
  // the last 8 k-tiles of row block i are the diagonal block W_ii: lower triangular (gemm_core.cuh, has_tri_stages)
  static constexpr int kTriMode = 1;
  __device__ __forceinline__ bool tri_diag() const { return kt >= i * KT_PER_BLOCK; }
  __device__ __forceinline__ int tri_g() const { return kt - i * KT_PER_BLOCK; }
  __device__ __forceinline__ void next() {
    if (kt == (i + 1) * KT_PER_BLOCK - 1) {
      ++j;
      i = zigzag_row(j, y, ns2);
      kt = 0;
    } else {
      ++kt;
    }
  }
};

// out[c] = (sum of the even rows of `in`, ascending) + (sum of the odd rows, ascending): the order in which the
// fused epilogue of score_trmm_kernel adds its per-warp-row running sums, so both paths give the same bits.
__global__ void __launch_bounds__(256) reduce_rows2_kernel(const double *__restrict__ in, int P, size_t ld,
                                                           double *__restrict__ out, int count) {
  const int c = blockIdx.x * 256 + threadIdx.x;
  if (c >= count) return;
  const double a0 = ordered_sum(in + c, 2 * ld, P / 2), a1 = ordered_sum(in + ld + c, 2 * ld, P / 2);   // P is even
  out[c] = a0 + a1;
}

// reduce_rows_kernel (mu partials) and reduce_rows2_kernel (sums of squares) of one slice in ONE launch, for the
// tiny-batch path where every launch is a visible share of the call: grid.y = 0 -> mu, 1 -> sums of squares
__global__ void __launch_bounds__(256) reduce_rows_pair_kernel(const double *__restrict__ in_mu, const double *__restrict__ in_ss,
                                                               int P, size_t ld, double *__restrict__ out_mu,
                                                               double *__restrict__ out_ss, int count) {
  const int c = blockIdx.x * 256 + threadIdx.x;
  if (c >= count) return;
  if (blockIdx.y == 0) {
    out_mu[c] = ordered_sum(in_mu + c, ld, P);
  } else {
    const double a0 = ordered_sum(in_ss + c, 2 * ld, P / 2), a1 = ordered_sum(in_ss + ld + c, 2 * ld, P / 2);
    out_ss[c] = a0 + a1;
  }
}

// Julia-order argmax of (v, i) pairs over the 256 threads of a CTA (i == LLONG_MAX: no candidate); result in sv[0], si[0].
__device__ __forceinline__ void block_argmax_256(double *sv, long long *si, double v, long long i) {
  const int tid = threadIdx.x;
  sv[tid] = v;
  si[tid] = i;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (tid < o) {
      const long long i2 = si[tid + o];
      if (i2 != 0x7fffffffffffffffLL && (si[tid] == 0x7fffffffffffffffLL || acq_better(sv[tid + o], i2, sv[tid], si[tid]))) {
        sv[tid] = sv[tid + o];
        si[tid] = i2;
      }
    }
    __syncthreads();
  }
}

// grid = (candidate blocks, ns row-block splits).  Each finished 128x128 tile of V = W K* contributes one
// partial column sum of squares per (row block, warp-row half); reduce_rows2_kernel adds them (unfused path).
__global__ void __launch_bounds__(GEMM_THREADS, 1) score_trmm_kernel(const __grid_constant__ ScoreParams p) {
  const int cb = blockIdx.x, y = blockIdx.y, ns2 = 2 * gridDim.y;
  ScoreIt it{p.W, p.Ks + (size_t)cb * p.ktiles * TILE_ELEMS, 0, zigzag_row(0, y, ns2), 0, p.nblk, p.ktiles, y, ns2};
  double *vt = p.VT ? p.VT + (size_t)cb * p.ktiles * TILE_ELEMS : nullptr;
  // fused: running column sums of squares per warp row, in the 4 KB scratch behind the ring ([2][128]; every slot is
  // owned by one lane, so no synchronisation is needed until the end) -- eight more live registers per thread in the
  // mainloop cost 3 % of its throughput
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  double *ssrun = reinterpret_cast<double *>(smem_raw + GEMM_RING_BYTES);
  if (p.fused && (threadIdx.x & 31) < 4) {
    const int w_ = threadIdx.x >> 5, l_ = threadIdx.x & 31;
#pragma unroll
    for (int fn = 0; fn < 4; ++fn) ssrun[(w_ >> 2) * 128 + 32 * (w_ & 3) + 8 * fn + 2 * l_] = ssrun[(w_ >> 2) * 128 + 32 * (w_ & 3) + 8 * fn + 2 * l_ + 1] = 0.0;
  }
  gemm_pipeline(it, it, [&](int tile, const double(&acc)[8][4][2], const FragCoord &fc) {
    if (vt) store_block(vt + (size_t)tile * KT_PER_BLOCK * TILE_ELEMS, true, 1.0, nullptr, acc, fc);
    double *dst = p.ss_part + (size_t)(2 * tile + fc.wm) * p.ld + (size_t)cb * 128 + 32 * fc.wn;
#pragma unroll
    for (int fn = 0; fn < 4; ++fn)
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        double v = 0.0;
#pragma unroll
        for (int fm = 0; fm < 8; ++fm) v = fma(acc[fm][fn][e], acc[fm][fn][e], v);
        v += __shfl_xor_sync(0xffffffffu, v, 4);
        v += __shfl_xor_sync(0xffffffffu, v, 8);
        v += __shfl_xor_sync(0xffffffffu, v, 16);
        if (fc.lane < 4) {
          if (p.fused)
            ssrun[fc.wm * 128 + 32 * fc.wn + 8 * fn + 2 * fc.lane + e] += v;
          else
            dst[8 * fn + 2 * fc.lane + e] = v;
        }
      }
  });
  if (!p.fused) return;
  // ---- fused epilogue: this CTA owns candidates cb*128 .. +127 of the chunk ----
  double *scr = reinterpret_cast<double *>(smem_raw);                 // argmax scratch (the ring is idle now)
  long long *sidx = reinterpret_cast<long long *>(smem_raw + 4096);
  const int tid = threadIdx.x;
  __syncthreads();   // every warp is through the ring and has added its last tile to ssrun
  // xcov's partial means of these 128 candidates: one coalesced sweep into the (idle) ring, summed in order below --
  // P dependent global loads per thread would hold the SM (and its tensor pipe) for tens of microseconds
  double *mup = reinterpret_cast<double *>(smem_raw + 8192);           // [P][128], P <= 2 * 64
  const int Pm = p.P < 128 ? p.P : 128;
  for (int e = tid; e < Pm * 128; e += GEMM_THREADS) mup[e] = p.mu_part[(size_t)(e >> 7) * p.ld + cb * 128 + (e & 127)];
  __syncthreads();
  double result = -INFINITY;
  long long ridx = 0x7fffffffffffffffLL;
  if (tid < 128) {
    const int c = cb * 128 + tid;
    const double ss = ssrun[tid] + ssrun[128 + tid];
    double mu = 0.0;
    for (int q = 0; q < Pm; ++q) mu += mup[q * 128 + tid];
    for (int q = Pm; q < p.P; ++q) mu += p.mu_part[(size_t)q * p.ld + c];
    p.ss_row[c] = ss;
    p.mu_row[c] = mu;
    const long long m = p.ap.m0 + c;
    if (c < p.ap.chunk && m < p.ap.M) {
      result = acq_candidate(p.ap, c, m);
      ridx = m;
    }
  }
  __syncthreads();   // scr is reused by the argmax
  if (p.ap.blk_val == nullptr) return;
  block_argmax_256(scr, sidx, result, ridx);
  __shared__ unsigned int s_last;
  if (tid == 0) {
    p.ap.blk_val[cb] = scr[0];
    p.ap.blk_idx[cb] = sidx[0];
    __threadfence();
    s_last = atomicAdd(p.counter, 1u) == gridDim.x - 1 ? 1u : 0u;
  }
  __syncthreads();
  if (!s_last) return;
  // last CTA of the launch: fold the block winners (fixed order) into the call's running winner
  __threadfence();
  double v = 0.0;
  long long ix = 0x7fffffffffffffffLL;
  for (int b = tid; b < (int)gridDim.x; b += 256) {
    const long long i2 = p.ap.blk_idx[b];
    if (i2 != 0x7fffffffffffffffLL && (ix == 0x7fffffffffffffffLL || acq_better(p.ap.blk_val[b], i2, v, ix))) {
      v = p.ap.blk_val[b];
      ix = i2;
    }
  }
  block_argmax_256(scr, sidx, v, ix);
  if (tid == 0) {
    if (sidx[0] != 0x7fffffffffffffffLL && (*p.bidx < 0 || acq_better(scr[0], sidx[0], *p.best, *p.bidx))) {
      *p.best = scr[0];
      *p.bidx = sidx[0];
    }
    *p.counter = 0u;
  }
}

// ---------------------------------------------------------------------------------------------
// full posterior covariance of a small candidate batch (cov / mean_and_cov, gaussian_process.jl:163-167,180-184)
//   cov[i][j] = k(x*_i, x*_j) - (V^T V)[i][j] + 1e-18 [i == j],   diagonal through _clip_var
// C = V^T V arrives tile-packed (lower block triangle computed; mirrored here so the result is exactly symmetric).
// ---------------------------------------------------------------------------------------------


// ---------------------------------------------------------------------------------------------
// device-side candidate generation: the batch never exists in host memory (SURVEY.md 8f rank 3)
//   grid     GridAM's Iterators.product of per-dimension ranges, first dimension fastest (grid.jl:30-43):
//            x_j = lo_j + step_j * ((m / prod_{i<j} count_i) mod count_j)
//   uniform  SamplingAM with a uniform prior over the box (sampling.jl:59-75): counter-based generator,
//            x_j = lb_j + u(seed, m, j) (ub_j - lb_j),  u = splitmix64(seed + (m*d + j) * golden) >> 11 * 2^-53
//            (stateless, so any shard of [0, M) reproduces the same points on any number of GPUs)
// ---------------------------------------------------------------------------------------------
struct CandGen {
  int mode;   // 0 = candidates supplied by the caller, 1 = grid, 2 = uniform box
  int d;
  double lo[32], step[32];      // grid origin / step, or box lower bound / width
  long long count[32];          // grid points per dimension
  unsigned long long seed;
  long long first;              // global index of the shard's first candidate (multi-GPU: contiguous index blocks)
};

__host__ __device__ __forceinline__ double splitmix_unit(unsigned long long seed, unsigned long long ctr) {
  unsigned long long z = seed + (ctr + 1ull) * 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  z = z ^ (z >> 31);
  return (double)(z >> 11) * (1.0 / 9007199254740992.0);
}

__host__ __device__ __forceinline__ double cand_coord(const CandGen &gq, long long m, int j) {
  if (gq.mode == 1) {
    long long r = m;
    for (int i = 0; i < j; ++i) r /= gq.count[i];
    return fma((double)(r % gq.count[j]), gq.step[j], gq.lo[j]);
  }
  // plain multiply-then-add (two roundings) so that any host language reproduces the points bit for bit
#ifdef __CUDA_ARCH__
  return __dadd_rn(gq.lo[j], __dmul_rn(splitmix_unit(gq.seed, (unsigned long long)m * gq.d + j), gq.step[j]));
#else
  volatile double t = splitmix_unit(gq.seed, (unsigned long long)m * gq.d + j) * gq.step[j];
  return gq.lo[j] + t;
#endif
}

__global__ void gen_candidates_kernel(CandGen gq, long long m0, int ch, double *xs) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= ch * gq.d) return;
  xs[e] = cand_coord(gq, gq.first + m0 + e / gq.d, e % gq.d);
}

// Scale + round training inputs once per fit: Xt[k][i] = round?(X[k*d+i]) * invl[i], zero padded.
__global__ void scale_train_kernel(const double *X, int d, int n, int n_pad, int DP, const double *invl,
                                   unsigned long long disc_bits, double *Xt) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n_pad * DP) return;
  const int k = e / DP, i = e % DP;
  double v = 0.0;
  if (k < n && i < d) {
    v = X[(size_t)k * d + i];
    if ((disc_bits >> i) & 1ull) v = rint(v);
    v *= invl[i];
  }
  Xt[e] = v;
}

}  // namespace boss
