// tk_small.cu -- warp-register batched log marginal likelihood for small training sets (n <= 32) and the
// covariance vector of boss_gp_append; instantiated for every (covariance function, padded input dimension).
//
// One warp per hyper-parameter sample; lane i owns row i of K in registers.  Kernel-matrix construction,
// right-looking Cholesky (pivot and column broadcast by warp shuffles), log-determinant and the forward
// substitution all happen in one pass over the columns -- K, L and w never exist in memory.  This is the
// regime of BASELINE config C1 (n = 20..30, d <= 2) and of the reference's unit tests (n = 3), where the
// fitters evaluate hundreds to thousands of hyper-parameter vectors per BO iteration
// (SamplingMAP src/model_fitters/sampling.jl:59-78, OptimizationMAP multistart optimization.jl:116-119,
// TuringBI ext/TuringExt.jl:78-86) and a 128-padded blocked factorisation would be almost all padding.
// Reference arithmetic: gp_data_loglike_slice (src/models/gaussian_process.jl:269-280) -> logpdf(::FiniteGP).
#include "common.cuh"
#include "tk_params.cuh"

namespace boss {

template <int KID, int DP>
__global__ void __launch_bounds__(SMALL_WARPS * 32) loglik_small_kernel(SmallLoglikParams p) {
  __shared__ double xs[SMALL_N * DP];   // raw (rounded) training inputs, zero padded to DP
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int e = tid; e < SMALL_N * DP; e += SMALL_WARPS * 32) {
    const int k = e / DP, q = e % DP;
    double v = 0.0;
    if (k < p.n && q < p.d) {
      v = p.X[(size_t)k * p.d + q];
      if ((p.disc_bits >> q) & 1ull) v = rint(v);
    }
    xs[e] = v;
  }
  __syncthreads();
  const long long s = (long long)blockIdx.x * SMALL_WARPS + warp;
  if (s >= p.S) return;
  const int n = p.n;

  // hyper-parameter conditioning (gaussian_process.jl:227-241)
  bool neg = false;
  double invl[DP];
#pragma unroll
  for (int q = 0; q < DP; ++q) {
    double l = 1.0;
    if (q < p.d) {
      l = p.ls[(size_t)s * p.d + q];
      if (!(l >= 0.0)) neg = true;
    }
    invl[q] = (q < p.d) ? 1.0 / (l + MIN_PARAM_VALUE) : 0.0;
  }
  const double a_raw = p.amp[s], s_raw = p.noise[s];
  if (!(a_raw >= 0.0) || !(s_raw >= 0.0)) neg = true;
  const double am = a_raw + MIN_PARAM_VALUE, sn = s_raw + MIN_PARAM_VALUE;
  const double a2 = am * am, s2 = sn * sn;

  // row `lane` of K: scaled coordinates are rounded products (x * (1/l)) exactly as in the blocked path
  double xi[DP];
#pragma unroll
  for (int q = 0; q < DP; ++q) xi[q] = __dmul_rn(xs[(lane < n ? lane : 0) * DP + q], invl[q]);
  double a[SMALL_N];
#pragma unroll
  for (int j = 0; j < SMALL_N; ++j) {
    double v = 0.0;
    if (j < n) {   // uniform
      double d2 = 0.0;
#pragma unroll
      for (int q = 0; q < DP; ++q) {
        const double df = xi[q] - __dmul_rn(xs[j * DP + q], invl[q]);
        d2 = fma(df, df, d2);
      }
      v = a2 * kappa<KID>(d2, p.rq_a);
      if (j == lane) v += s2;
    }
    a[j] = v;
  }
  double y = (lane < n) ? p.ymm[(size_t)s * p.ldy + lane] : 0.0;

  // right-looking Cholesky + forward substitution, one column per step
  bool bad = false;
  double logdet = 0.0, mahal = 0.0;
#pragma unroll
  for (int k = 0; k < SMALL_N; ++k) {
    if (k < n) {   // uniform
      double piv = __shfl_sync(0xffffffffu, a[k], k);
      if (!(piv > 0.0)) {   // LAPACK dpotrf info > 0 (also NaN)
        bad = true;
        piv = 1.0;
      }
      const double lkk = sqrt(piv);
      const double inv = 1.0 / lkk;
      logdet += log(lkk);
      const double lik = (lane > k) ? a[k] * inv : 0.0;     // L[lane][k] below the diagonal
      const double wk = __shfl_sync(0xffffffffu, y, k) * inv;
      mahal = fma(wk, wk, mahal);
      y = fma(-lik, wk, y);
#pragma unroll
      for (int j = k + 1; j < SMALL_N; ++j) {
        if (j < n) {
          const double ljk = __shfl_sync(0xffffffffu, lik, j);
          a[j] = fma(-lik, ljk, a[j]);                      // only lanes >= j hold live entries
        }
      }
    }
  }
  if (lane == 0) {
    double ll = -((double)n * 1.8378770664093453 + 2.0 * logdet + mahal) * 0.5;
    if (bad) ll = -INFINITY;
    if (neg) ll = NAN;
    p.loglik[s] = ll;
  }
}

// k[i] = a^2 kappa(|x~_i - x~+|), i < n (zero beyond); also appends the scaled point as row n of Xt.
template <int KID, int DP>
__global__ void append_kvec_kernel(const double *xnew, int d, int n, int n_pad, const double *invl,
                                   unsigned long long disc_bits, double a2, double rq_a, double *Xt,
                                   double *kvec) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_pad) return;
  double xn[DP];
  load_scaled_point<DP>(xn, xnew, d, invl, disc_bits, true);
  double val = 0.0;
  if (i < n) {
    double d2 = 0.0;
#pragma unroll
    for (int q = 0; q < DP; ++q) {
      const double df = Xt[(size_t)i * DP + q] - xn[q];
      d2 = fma(df, df, d2);
    }
    val = a2 * kappa<KID>(d2, rq_a);
  }
  kvec[i] = val;
  if (i == n) {
#pragma unroll
    for (int q = 0; q < DP; ++q) Xt[(size_t)n * DP + q] = xn[q];
  }
}

bool launch_loglik_small(int kid, int dp, const SmallLoglikParams &p, int nblocks, cudaStream_t st) {
#define CALL(K, D) loglik_small_kernel<K, D><<<nblocks, SMALL_WARPS * 32, 0, st>>>(p)
  BOSS_DISPATCH_KID_DP(CALL, kid, dp)
#undef CALL
}
bool launch_append_kvec(int kid, int dp, const double *xnew, int d, int n, int n_pad, const double *invl,
                        unsigned long long disc_bits, double a2, double rq_a, double *Xt, double *kvec, cudaStream_t st) {
#define CALL(K, D) append_kvec_kernel<K, D><<<(n_pad + 255) / 256, 256, 0, st>>>(xnew, d, n, n_pad, invl, disc_bits, a2, rq_a, Xt, \
                                                                             kvec)
  BOSS_DISPATCH_KID_DP(CALL, kid, dp)
#undef CALL
}

}  // namespace boss
