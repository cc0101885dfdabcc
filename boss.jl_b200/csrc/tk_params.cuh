// tk_params.cuh -- parameter blocks and host launchers of the kernels that are templated on
// (covariance function KID, padded input dimension DP).  Those 7 kernel families x 35 instantiations are most of the
// library's compile time, so they live in their own translation units (tk_build.cu, tk_score.cu, tk_small.cu) and are
// reached through the plain launch_* functions declared at the end of this file.
#pragma once
#include "acq.cuh"

namespace boss {

struct BuildKParams {
  const double *X;          // d x n raw training inputs (shared by all samples)
  int d, n, nblk, ktiles;   // nblk = n_pad/128, ktiles = n_pad/16
  const double *ls;         // d x S raw length-scales
  const double *amp;        // S raw amplitudes
  const double *noise;      // S raw noise std
  unsigned long long disc_bits;
  double *K;                // S matrices, P-layout, stride K_stride
  size_t K_stride;
  int *status;              // S; set to -1 on negative hyper-parameters (reference asserts)
  int skip_diag;            // diagonal tiles are produced elsewhere (potrf_fused_kernel generates K_jj on chip)
  double rq_a;              // RationalQuadratic shape parameter (KID 4; ignored by the other kernels)
};

struct LlGradParams {
  const double *X;
  int d, n, nblk, ktiles;
  const double *ls, *amp, *noise;   // raw hyper-parameters of the sub-batch
  unsigned long long disc_bits;
  const double *Kinv;
  size_t K_stride;
  const double *alpha;   // [S][n_pad]
  double *part;          // [S][ntiles][DP + 2]
  double rq_a;
};

struct XcovParams {
  const double *Xs;        // d x . raw candidates (device), candidate m at column (m - in_off)
  long long M, m0, in_off; // global count, first candidate of this chunk
  int d, n, n_pad, ktiles;
  const double *Xt;        // [n_pad][DP] scaled (and rounded) training inputs
  const double *invl;      // [DP]
  unsigned long long disc_bits;
  const double *alpha;     // [n_pad] K^-1 (y - m), zero padded
  double a2;
  double *Ks;              // chunk scratch, P-layout: rows = candidates of the chunk, cols = training index
  double *mu_part;         // [2*nblk][ld] per-(128-chunk of training points, k-half) partials of K*^T alpha
  int ld;                  // leading dimension of mu_part (= chunk capacity)
  double rq_a;
};

constexpr int XCOV_KC = 128;  // training points staged per shared-memory pass

// The FP32 mean tier of argmax screening (DESIGN.md 2.9): mu~ with a proven bound E on |mu~ - mu|, from per-call FP32
// copies of the centred training inputs and of alpha (screen_consts_kernel), and the bound verdicts of the candidates
// (screen_mean_bound_kernel in tk_score.cu).  One launch covers every slice of a call, up to SCREEN_F32_MAX_SL of them,
// all of one covariance function.
struct ScreenSlice {
  const float4 *tfrag;   // [n_pad / 8][KP / 8][32] per eight-point tile, k-step and lane: the MMA's B fragments of the
                         // centred training inputs t~ = fp32(ut - c), TF32-split: (b0 hi, b1 hi, b0 lo, b1 lo)
  const float4 *tn_al;   // [n_pad / 2] (|t~_j|^2, |t~_j+1|^2, alpha_j, alpha_j+1) rounded to FP32, j even
  const double *A;       // [SCREEN_NCONST] A1 = sum |alpha_j|, A3 = sum |alpha_j| |ut_j - c|^2, the centre c (DP)
  const double *invl;    // [DP]
  unsigned long long disc_bits;
  double a2;
  int n_pad;
};
constexpr int SCREEN_F32_MAX_SL = 16;
struct ScreenF32Params {
  const double *Xs;       // d x . raw candidates (device), candidate m at column (m - in_off)
  long long m0, M, in_off;   // candidates [m0, M)
  int d, nsl;
  ScreenSlice sl[SCREEN_F32_MAX_SL];
  AcqParams hi, lo;       // the bound pass at mu~ + E' and at mu~ - E' (mu / sumsq unused; hi.acq, lo.acq get the bounds)
  double thr;             // a candidate survives unless its hi bound is below thr
  long long *cnt;         // survivors per 128 candidates, or null: the bounds only
  double *mu_out, *e_out; // or [nsl][ld] indexed by m - m0: mu~ and E instead of the bounds
  int ld;
};
constexpr int SCREEN_NCONST = 2 + 32;
// E = a^2 2^-24 (SCREEN_C_EVAL A1 + L2 k (|u - c|^2 A1 + A3))   (DESIGN.md 2.9), L2 = sup |d kappa / d(d2)|, and
// k 2^-24 (|u - c|^2 + |ut_j - c|^2) bounds the error of the tensor-core d2 with KP = DP rounded up to 8
constexpr double SCREEN_C_EVAL = 64.0;
__host__ __device__ constexpr double screen_l2(int kid) { return kid == 0 ? 0.5 : kid == 1 ? 1.5 : 5.0 / 6.0; }
__host__ __device__ constexpr double screen_k_dot(int dp) { return 24.0 + 7.5 * (8 * ((dp + 7) / 8)); }

struct CovFinishParams {
  const double *Xs;     // d x M raw candidates
  int M, d, ktilesC;    // ktilesC = M_pad / 16
  const double *invl;
  unsigned long long disc_bits;
  double a2;
  const double *C;      // P-layout M_pad x M_pad
  const double *mu;     // [M] K*^T alpha
  const double *prior_mean;  // [M] or null
  double *mu_out;       // [M] or null
  double *cov;          // M x M column-major
  int *any_fail;
  double rq_a;
};

struct GradParams {
  const double *Xs;
  long long M, m0, in_off;
  int d, n, n_pad, ktiles, chunk_ld;
  const double *Xt, *invl, *alpha;
  unsigned long long disc_bits;
  double a2;
  const double *UT;    // chunk scratch (P-layout), u = K^-1 k*
  double *gm_part, *gv_part;  // [2*nblk][d][chunk_ld] per-(training chunk, k-half) partial sums (unscaled)
  double rq_a;
};

constexpr int SMALL_N = 32;
constexpr int SMALL_WARPS = 8;

struct SmallLoglikParams {
  const double *X;      // d x n raw training inputs (shared)
  int d, n;
  const double *ymm;    // n (ldy = 0) or per sample at ymm + s*ldy
  long long ldy;
  const double *ls;     // d x S raw length-scales
  const double *amp, *noise;  // S each, raw
  unsigned long long disc_bits;
  long long S;
  double *loglik;       // S: value, -Inf (not positive definite) or NaN (negative hyper-parameter)
  double rq_a;
};

// ---- host launchers: dispatch on (KID 0..4, dp in {2,4,6,8,12,16,32}); false = unsupported combination ----
// KIDs: 0 SqExponential, 1 Matern32, 2 Matern52, 3 Matern12, 4 RationalQuadratic (kernel_fn.cuh).  The FP32 mean tier
// (launch_screen_mean_bound) exists for KIDs 0-2 only: its error bound needs sup |d kappa / d(d2)|, which is infinite for
// Matern12 and not derived for RQ's FP32 evaluation, so those kernels screen with FP64 means (DESIGN.md 2.14).
constexpr int NUM_KID = 5;
__host__ __device__ constexpr bool kid_has_f32_tier(int kid) { return kid >= 0 && kid <= 2; }
bool launch_build_k(int kid, int dp, const BuildKParams &p, dim3 grid, cudaStream_t st);
bool launch_loglik_grad_tile(int kid, int dp, const LlGradParams &p, dim3 grid, cudaStream_t st);
bool launch_xcov(int kid, int dp, const XcovParams &p, dim3 grid, cudaStream_t st);
bool launch_xcov_mean(int kid, int dp, const XcovParams &p, dim3 grid, cudaStream_t st);   // mu partials only (p.Ks unused)
size_t screen_mean_bound_smem(int dp, int nsl);   // dynamic shared memory of one CTA
bool launch_screen_mean_bound(int kid, int dp, const ScreenF32Params &p, int nblocks, cudaStream_t st);
bool launch_kappa_f32_sweep(int kid, const double *r, int n, double *out, cudaStream_t st);
bool launch_mma_d2(int dp, const float *u, const float *t, const float *nu, const float *nt, int mt, int nt_, float *d2,
                   cudaStream_t st);
bool launch_cov_finish(int kid, int dp, const CovFinishParams &p, dim3 grid, cudaStream_t st);
bool launch_grad(int kid, int dp, const GradParams &p, dim3 grid, cudaStream_t st);
bool launch_loglik_small(int kid, int dp, const SmallLoglikParams &p, int nblocks, cudaStream_t st);
bool launch_append_kvec(int kid, int dp, const double *xnew, int d, int n, int n_pad, const double *invl,
                        unsigned long long disc_bits, double a2, double rq_a, double *Xt, double *kvec, cudaStream_t st);

#define BOSS_DISPATCH_DP_CASES(CALL, K)  \
  case (K) * 100 + 2: CALL(K, 2); return true;     \
  case (K) * 100 + 4: CALL(K, 4); return true;     \
  case (K) * 100 + 6: CALL(K, 6); return true;     \
  case (K) * 100 + 8: CALL(K, 8); return true;     \
  case (K) * 100 + 12: CALL(K, 12); return true;   \
  case (K) * 100 + 16: CALL(K, 16); return true;   \
  case (K) * 100 + 32: CALL(K, 32); return true;

#define BOSS_DISPATCH_KID_DP(CALL, kid, dp) \
  switch ((kid) * 100 + (dp)) {             \
    BOSS_DISPATCH_DP_CASES(CALL, 0)         \
    BOSS_DISPATCH_DP_CASES(CALL, 1)         \
    BOSS_DISPATCH_DP_CASES(CALL, 2)         \
    BOSS_DISPATCH_DP_CASES(CALL, 3)         \
    BOSS_DISPATCH_DP_CASES(CALL, 4)         \
    default: return false;                  \
  }

// the kernels of the FP32 mean tier: KIDs 0-2 only (see kid_has_f32_tier)
#define BOSS_DISPATCH_KID_DP_F32(CALL, kid, dp) \
  switch ((kid) * 100 + (dp)) {                 \
    BOSS_DISPATCH_DP_CASES(CALL, 0)             \
    BOSS_DISPATCH_DP_CASES(CALL, 1)             \
    BOSS_DISPATCH_DP_CASES(CALL, 2)             \
    default: return false;                      \
  }

}  // namespace boss
