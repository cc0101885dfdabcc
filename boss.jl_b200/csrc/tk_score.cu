// tk_score.cu -- the FP64-pipe kernels of the scoring path that evaluate the covariance function: cross-covariance
// K*^T + posterior mean (row a3), the finish of the full posterior covariance, and the kernel derivatives of the
// x-gradient (row g1); instantiated for every (covariance function, padded input dimension).
#include "common.cuh"
#include "tk_params.cuh"

namespace boss {

// grid = (candidate blocks, splits over the 128-point training chunks).  Every chunk's contribution to
// mu is written as its own partial (fixed summation order downstream), so results do not depend on the split.
// STORE_KS = false: the mean partials only (argmax screening needs mu, not K*^T); same partials, same bits.
template <int KID, int DP, bool STORE_KS = true>
__global__ void __launch_bounds__(256) xcov_kernel(XcovParams p) {
  __shared__ double xt[XCOV_KC * DP];
  __shared__ double al[XCOV_KC];
  __shared__ double etab[EXPTAB_N];
  exptab_init(etab);
  const int tid = threadIdx.x, r = tid & 127, kh = tid >> 7;
  const int cb = blockIdx.x;
  const long long m = p.m0 + (long long)cb * 128 + r;
  double xc[DP];
  load_scaled_point<DP>(xc, p.Xs + (size_t)(m - p.in_off) * p.d, p.d, p.invl, p.disc_bits, m < p.M);

  double *rowbase = p.Ks + (size_t)cb * p.ktiles * TILE_ELEMS + (((r >> 3) << 1) << 6) + ((r & 7) << 3);
  for (int k0 = blockIdx.y * XCOV_KC; k0 < p.n_pad; k0 += gridDim.y * XCOV_KC) {
    double mu_acc = 0.0;
    __syncthreads();
    for (int e = tid; e < XCOV_KC * DP; e += 256) xt[e] = p.Xt[(size_t)k0 * DP + e];
    if (tid < XCOV_KC) al[tid] = p.alpha[k0 + tid];
    __syncthreads();
    // the last chunk may run past n: its padded columns must be exactly 0 (W is identity there)
    const int live = p.n - k0;
    for (int mcol = kh; mcol < XCOV_KC / 8; mcol += 2) {
      double v[8];
#pragma unroll
      for (int kk = 0; kk < 8; ++kk) {   // eight independent, branch-free chains: the scheduler interleaves them
        const int kl = mcol * 8 + kk;
        double d2 = 0.0;
#pragma unroll
        for (int i = 0; i < DP; ++i) {
          const double df = xc[i] - xt[kl * DP + i];
          d2 = fma(df, df, d2);
        }
        v[kk] = p.a2 * kappa_fast<KID>(d2, etab);
      }
      if (live < XCOV_KC) {
#pragma unroll
        for (int kk = 0; kk < 8; ++kk) v[kk] = (mcol * 8 + kk < live) ? v[kk] : 0.0;
      }
#pragma unroll
      for (int kk = 0; kk < 8; ++kk) mu_acc = fma(v[kk], al[mcol * 8 + kk], mu_acc);
      if (!STORE_KS) continue;
      const int kg = k0 + mcol * 8;  // global training index of v[0]
      double *dst = rowbase + (size_t)(kg >> 4) * TILE_ELEMS + (((kg >> 3) & 1) << 6);
#pragma unroll
      for (int q = 0; q < 4; ++q) *reinterpret_cast<double2 *>(dst + 2 * q) = make_double2(v[q], v[q + 4]);
    }
    p.mu_part[(size_t)(2 * (k0 / XCOV_KC) + kh) * p.ld + (size_t)cb * 128 + r] = mu_acc;
  }
}

// The FP32 mean tier of argmax screening (DESIGN.md 2.9): xcov_kernel<KID, DP, false>'s grid, partial layout and
// reduction order, with the distances and kappa in FP32 (packed f32x2 differences, MUFU rsqrt / ex2).  Each run of 8
// training points is summed in FP32 and added to an FP64 accumulator (one conversion per 8 pairs).  Blocks of split 0
// also write each candidate's error bound E (tk_params.cuh), from |u| in FP64 and the per-call constants A1, A2.
template <int KID, int DP>
__global__ void __launch_bounds__(256) xcov_mean_f32_kernel(XcovF32Params q) {
  static_assert(DP % 2 == 0, "padded dimensions are even");
  const XcovParams &p = q.x;
  __shared__ float2 xt[XCOV_KC * DP / 2];
  __shared__ float al[XCOV_KC];
  const int tid = threadIdx.x, r = tid & 127, kh = tid >> 7;
  const int cb = blockIdx.x;
  const long long m = p.m0 + (long long)cb * 128 + r;
  float2 xc[DP / 2];
  {
    double x64[DP];
    load_scaled_point<DP>(x64, p.Xs + (size_t)(m - p.in_off) * p.d, p.d, p.invl, p.disc_bits, m < p.M);
    double n2 = 0.0;
#pragma unroll
    for (int i = 0; i < DP; ++i) n2 = fma(x64[i], x64[i], n2);
#pragma unroll
    for (int i = 0; i < DP / 2; ++i) xc[i] = make_float2((float)x64[2 * i], (float)x64[2 * i + 1]);
    if (blockIdx.y == 0 && kh == 0)
      q.E[(size_t)cb * 128 + r] =
          p.a2 * 0x1p-24 * (SCREEN_C_EVAL * q.A[0] + SCREEN_L_KAPPA * fma(sqrt(n2), q.A[0], q.A[1]));
  }
  const float2 *xg = reinterpret_cast<const float2 *>(q.Xt_neg);
  for (int k0 = blockIdx.y * XCOV_KC; k0 < p.n_pad; k0 += gridDim.y * XCOV_KC) {
    double mu_acc = 0.0;
    __syncthreads();
    for (int e = tid; e < XCOV_KC * DP / 2; e += 256) xt[e] = xg[(size_t)k0 * (DP / 2) + e];
    if (tid < XCOV_KC) al[tid] = q.alpha[k0 + tid];
    __syncthreads();
    for (int mcol = kh; mcol < XCOV_KC / 8; mcol += 2) {
      float s8 = 0.0f;
#pragma unroll
      for (int kk = 0; kk < 8; ++kk) {   // eight independent chains; padded columns have alpha = 0 and Xt = 0
        const int kl = mcol * 8 + kk;
        float2 acc = make_float2(0.0f, 0.0f);
#pragma unroll
        for (int i = 0; i < DP / 2; ++i) {
          const float2 df = __fadd2_rn(xc[i], xt[kl * (DP / 2) + i]);
          acc = __ffma2_rn(df, df, acc);
        }
        s8 = fmaf(al[kl], kappa_f32<KID>(acc.x + acc.y), s8);
      }
      mu_acc += (double)s8;
    }
    p.mu_part[(size_t)(2 * (k0 / XCOV_KC) + kh) * p.ld + (size_t)cb * 128 + r] = p.a2 * mu_acc;
  }
}

// FP32 kappa at d2 = r^2 (rounded to FP32) for the error-bound sweep of the tests
template <int KID>
__global__ void kappa_f32_sweep_kernel(const double *r, int n, double *out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = (double)kappa_f32<KID>((float)(r[i] * r[i]));
}

// full posterior covariance of a small candidate batch (cov / mean_and_cov, gaussian_process.jl:163-167,180-184)
//   cov[i][j] = k(x*_i, x*_j) - (V^T V)[i][j] + 1e-18 [i == j],   diagonal through _clip_var
template <int KID, int DP>
__global__ void __launch_bounds__(256) cov_finish_kernel(CovFinishParams p) {
  __shared__ double etab[EXPTAB_N];
  exptab_init(etab);
  __syncthreads();
  const int i = blockIdx.x * 16 + (threadIdx.x & 15), j = blockIdx.y * 16 + (threadIdx.x >> 4);
  if (i >= p.M || j >= p.M) return;
  double xi[DP], xj[DP];
  load_scaled_point<DP>(xi, p.Xs + (size_t)i * p.d, p.d, p.invl, p.disc_bits, true);
  load_scaled_point<DP>(xj, p.Xs + (size_t)j * p.d, p.d, p.invl, p.disc_bits, true);
  double d2 = 0.0;
#pragma unroll
  for (int q = 0; q < DP; ++q) {
    const double df = xi[q] - xj[q];
    d2 = fma(df, df, d2);
  }
  const int hi = max(i, j), lo = min(i, j);
  double v = p.a2 * kappa_fast<KID>(d2, etab) - p.C[p_index(hi, lo, p.ktilesC)];
  if (i == j) {
    v += VAR_JITTER;
    if (!clip_var(v)) *p.any_fail = 1;
    if (p.mu_out) p.mu_out[i] = p.prior_mean ? p.prior_mean[i] + p.mu[i] : p.mu[i];
  }
  p.cov[(size_t)j * p.M + i] = v;
}

// d mu / dx and d var / dx for one slice and one chunk (see grad.cuh).
template <int KID, int DP>
__global__ void __launch_bounds__(256) grad_kernel(GradParams p) {
  __shared__ double xt[XCOV_KC * DP];
  __shared__ double al[XCOV_KC];
  __shared__ double etab[EXPTAB_N];
  exptab_init(etab);
  const int tid = threadIdx.x, r = tid & 127, kh = tid >> 7;
  const int cb = blockIdx.x;
  const long long m = p.m0 + (long long)cb * 128 + r;
  double xc[DP];
  load_scaled_point<DP>(xc, p.Xs + (size_t)(m - p.in_off) * p.d, p.d, p.invl, p.disc_bits, m < p.M);
  const double *rowbase = p.UT + (size_t)cb * p.ktiles * TILE_ELEMS + (((r >> 3) << 1) << 6) + ((r & 7) << 3);
  for (int k0 = blockIdx.y * XCOV_KC; k0 < p.n_pad; k0 += gridDim.y * XCOV_KC) {
    double gm[DP], gv[DP];
#pragma unroll
    for (int i = 0; i < DP; ++i) gm[i] = gv[i] = 0.0;
    __syncthreads();
    for (int e = tid; e < XCOV_KC * DP; e += 256) xt[e] = p.Xt[(size_t)k0 * DP + e];
    if (tid < XCOV_KC) al[tid] = p.alpha[k0 + tid];
    __syncthreads();
    for (int mcol = kh; mcol < XCOV_KC / 8; mcol += 2) {
      const int kg = k0 + mcol * 8;
      const double *src = rowbase + (size_t)(kg >> 4) * TILE_ELEMS + (((kg >> 3) & 1) << 6);
      double u[8];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const double2 v = *reinterpret_cast<const double2 *>(src + 2 * q);
        u[q] = v.x;
        u[q + 4] = v.y;
      }
      double gk[8];
#pragma unroll
      for (int kk = 0; kk < 8; ++kk) {   // independent, branch-free chains
        const int kl = mcol * 8 + kk;
        double d2 = 0.0;
#pragma unroll
        for (int i = 0; i < DP; ++i) {
          const double df = xc[i] - xt[kl * DP + i];
          d2 = fma(df, df, d2);
        }
        gk[kk] = p.a2 * kappa_dr_over_r_fast<KID>(d2, etab);
      }
      if (p.n - k0 < XCOV_KC) {
#pragma unroll
        for (int kk = 0; kk < 8; ++kk) gk[kk] = (k0 + mcol * 8 + kk < p.n) ? gk[kk] : 0.0;
      }
#pragma unroll
      for (int kk = 0; kk < 8; ++kk) {
        const int kl = mcol * 8 + kk;
        const double t1 = gk[kk] * al[kl], t2 = gk[kk] * u[kk];
#pragma unroll
        for (int i = 0; i < DP; ++i) {
          const double df = xc[i] - xt[kl * DP + i];
          gm[i] = fma(t1, df, gm[i]);
          gv[i] = fma(t2, df, gv[i]);
        }
      }
    }
    const size_t prow = (size_t)(2 * (k0 / XCOV_KC) + kh) * p.d;
#pragma unroll
    for (int i = 0; i < DP; ++i) {
      if (i < p.d) {
        p.gm_part[(prow + i) * p.chunk_ld + cb * 128 + r] = gm[i];
        p.gv_part[(prow + i) * p.chunk_ld + cb * 128 + r] = gv[i];
      }
    }
  }
}

bool launch_xcov(int kid, int dp, const XcovParams &p, dim3 grid, cudaStream_t st) {
#define CALL(K, D) xcov_kernel<K, D><<<grid, 256, 0, st>>>(p)
  BOSS_DISPATCH_KID_DP(CALL, kid, dp)
#undef CALL
}
bool launch_xcov_mean(int kid, int dp, const XcovParams &p, dim3 grid, cudaStream_t st) {
#define CALL(K, D) xcov_kernel<K, D, false><<<grid, 256, 0, st>>>(p)
  BOSS_DISPATCH_KID_DP(CALL, kid, dp)
#undef CALL
}
bool launch_xcov_mean_f32(int kid, int dp, const XcovF32Params &p, dim3 grid, cudaStream_t st) {
#define CALL(K, D) xcov_mean_f32_kernel<K, D><<<grid, 256, 0, st>>>(p)
  BOSS_DISPATCH_KID_DP(CALL, kid, dp)
#undef CALL
}
bool launch_kappa_f32_sweep(int kid, const double *r, int n, double *out, cudaStream_t st) {
  const int nb = (n + 255) / 256;
  if (n < 1) return true;
  if (kid == 0) kappa_f32_sweep_kernel<0><<<nb, 256, 0, st>>>(r, n, out);
  else if (kid == 1) kappa_f32_sweep_kernel<1><<<nb, 256, 0, st>>>(r, n, out);
  else if (kid == 2) kappa_f32_sweep_kernel<2><<<nb, 256, 0, st>>>(r, n, out);
  else return false;
  return true;
}
bool launch_cov_finish(int kid, int dp, const CovFinishParams &p, dim3 grid, cudaStream_t st) {
#define CALL(K, D) cov_finish_kernel<K, D><<<grid, 256, 0, st>>>(p)
  BOSS_DISPATCH_KID_DP(CALL, kid, dp)
#undef CALL
}
bool launch_grad(int kid, int dp, const GradParams &p, dim3 grid, cudaStream_t st) {
#define CALL(K, D) grad_kernel<K, D><<<grid, 256, 0, st>>>(p)
  BOSS_DISPATCH_KID_DP(CALL, kid, dp)
#undef CALL
}

}  // namespace boss
