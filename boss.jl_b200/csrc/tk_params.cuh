// tk_params.cuh -- parameter blocks and host launchers of the kernels that are templated on
// (covariance function KID, padded input dimension DP).  Those 7 kernel families x 21 instantiations are most of the
// library's compile time, so they live in their own translation units (tk_build.cu, tk_score.cu, tk_small.cu) and are
// reached through the plain launch_* functions declared at the end of this file.
#pragma once
#include "kernel_fn.cuh"

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
};

constexpr int XCOV_KC = 128;  // training points staged per shared-memory pass

// The FP32 mean tier of argmax screening (DESIGN.md 2.9): mu~ with a proven bound E on |mu~ - mu|, from an FP32 copy
// of the training inputs and weights.  x.Xt / x.alpha are unused; x.mu_part receives the partials (FP64, same layout).
struct XcovF32Params {
  XcovParams x;
  const float *Xt_neg;   // [n_pad][DP] -(scaled training inputs), rounded to FP32
  const float *alpha;    // [n_pad] alpha rounded to FP32
  const double *A;       // [2] A1 = sum |alpha_j|, A2 = sum |alpha_j| |ut_j|  (screen_consts_kernel)
  double *E;             // [ld] the error bound of each candidate's mean
};
// E = a^2 2^-24 (SCREEN_C_EVAL A1 + SCREEN_L_KAPPA (|u| A1 + A2))   (DESIGN.md 2.9)
constexpr double SCREEN_C_EVAL = 64.0;
constexpr double SCREEN_L_KAPPA = 0.65;

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
};

// ---- host launchers: dispatch on (kernel_id 0..2, dp in {2,4,6,8,12,16,32}); false = unsupported combination ----
bool launch_build_k(int kid, int dp, const BuildKParams &p, dim3 grid, cudaStream_t st);
bool launch_loglik_grad_tile(int kid, int dp, const LlGradParams &p, dim3 grid, cudaStream_t st);
bool launch_xcov(int kid, int dp, const XcovParams &p, dim3 grid, cudaStream_t st);
bool launch_xcov_mean(int kid, int dp, const XcovParams &p, dim3 grid, cudaStream_t st);   // mu partials only (p.Ks unused)
bool launch_xcov_mean_f32(int kid, int dp, const XcovF32Params &p, dim3 grid, cudaStream_t st);
bool launch_kappa_f32_sweep(int kid, const double *r, int n, double *out, cudaStream_t st);
bool launch_cov_finish(int kid, int dp, const CovFinishParams &p, dim3 grid, cudaStream_t st);
bool launch_grad(int kid, int dp, const GradParams &p, dim3 grid, cudaStream_t st);
bool launch_loglik_small(int kid, int dp, const SmallLoglikParams &p, int nblocks, cudaStream_t st);
bool launch_append_kvec(int kid, int dp, const double *xnew, int d, int n, int n_pad, const double *invl,
                        unsigned long long disc_bits, double a2, double *Xt, double *kvec, cudaStream_t st);

#define BOSS_DISPATCH_KID_DP(CALL, kid, dp)       \
  switch ((kid) * 100 + (dp)) {                   \
    case 2: CALL(0, 2); return true;              \
    case 4: CALL(0, 4); return true;              \
    case 6: CALL(0, 6); return true;              \
    case 8: CALL(0, 8); return true;              \
    case 12: CALL(0, 12); return true;            \
    case 16: CALL(0, 16); return true;            \
    case 32: CALL(0, 32); return true;            \
    case 102: CALL(1, 2); return true;            \
    case 104: CALL(1, 4); return true;            \
    case 106: CALL(1, 6); return true;            \
    case 108: CALL(1, 8); return true;            \
    case 112: CALL(1, 12); return true;           \
    case 116: CALL(1, 16); return true;           \
    case 132: CALL(1, 32); return true;           \
    case 202: CALL(2, 2); return true;            \
    case 204: CALL(2, 4); return true;            \
    case 206: CALL(2, 6); return true;            \
    case 208: CALL(2, 8); return true;            \
    case 212: CALL(2, 12); return true;           \
    case 216: CALL(2, 16); return true;           \
    case 232: CALL(2, 32); return true;           \
    default: return false;                        \
  }

}  // namespace boss
