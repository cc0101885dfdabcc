// grad.cuh -- analytic x-gradients of the acquisition for the multi-start optimiser
// (reference: OptimizationAM pushes ForwardDiff.Dual candidates through the whole posterior stack,
//  src/acquisition_maximizers/optimization.jl:36,100-113; here the same derivative in closed form).
//
//   mu(x)    = m(x) + sum_k alpha_k k(x, x_k)         d mu  = sum_k alpha_k dk_k
//   var(x)   = a^2 - |W k*(x)|^2                       d var = -2 sum_k u_k dk_k ,  u = W^T (W k*) = K^-1 k*
//   dk_k/dx_j = a^2 kappa'(r)/r * (x~_j - x~_kj) / l_j
//
// Pipeline per chunk and slice: xcov -> score_trmm (also stores V^T) -> wtv_kernel (U^T = (W^T V)^T, the
// second triangular product, same DMMA mainloop) -> grad_kernel (kernel derivatives, FP64 pipe) ->
// acq_grad_kernel (chain rule through EI x PoF, or through the Monte-Carlo EI of a MixParams expression), or
// predict_grad_kernel (boss_gp_predict_grad: mu, var and their gradients themselves, in the caller's layout).
#pragma once
#include "score.cuh"

namespace boss {

// U[k][c] = sum_{r >= k} WT[k][r] V[r][c] ;  A = WT row block i (tiles 8i .. ktiles-1), B = V^T block of the CTA
struct WtvParams {
  const double *WT;
  const double *VT;   // chunk scratch: rows = candidates, cols = V row index
  double *UT;         // chunk scratch: rows = candidates, cols = training index
  int nblk, ktiles;
};
struct WtvIt {
  const double *wt;      // W^T (upper triangular): row block i uses k-tiles 8i .. ktiles-1
  const double *vt;
  int j, i, kt, nblk, ktiles, y, ns2;
  __device__ __forceinline__ bool valid() const { return i < nblk; }
  __device__ __forceinline__ const double *A() const { return wt + ((size_t)i * ktiles + kt) * TILE_ELEMS; }
  __device__ __forceinline__ const double *B() const { return vt + (size_t)kt * TILE_ELEMS; }
  __device__ __forceinline__ bool tile_end() const { return kt == ktiles - 1; }
  __device__ __forceinline__ int tile() const { return i; }
  // the first 8 k-tiles of row block i are the diagonal block W_ii^T: upper triangular (gemm_core.cuh, has_tri_stages)
  static constexpr int kTriMode = 2;
  __device__ __forceinline__ bool tri_diag() const { return kt < (i + 1) * KT_PER_BLOCK; }
  __device__ __forceinline__ int tri_g() const { return kt - i * KT_PER_BLOCK; }
  __device__ __forceinline__ void next() {
    if (kt == ktiles - 1) {
      ++j;
      i = zigzag_row(j, y, ns2);
      kt = i * KT_PER_BLOCK;
    } else {
      ++kt;
    }
  }
};
// grid = (candidate blocks, ns row-block splits), same zig-zag deal as score_trmm_kernel
__global__ void __launch_bounds__(GEMM_THREADS, 1) wtv_kernel(WtvParams p) {
  const int cb = blockIdx.x, y = blockIdx.y, ns2 = 2 * gridDim.y;
  const int i0 = zigzag_row(0, y, ns2);
  WtvIt it{p.WT, p.VT + (size_t)cb * p.ktiles * TILE_ELEMS, 0, i0, i0 * KT_PER_BLOCK, p.nblk, p.ktiles, y, ns2};
  double *ut = p.UT + (size_t)cb * p.ktiles * TILE_ELEMS;
  gemm_pipeline(it, it, [&](int tile, const double(&acc)[8][4][2], const FragCoord &fc) {
    store_block(ut + (size_t)tile * KT_PER_BLOCK * TILE_ELEMS, true, 1.0, nullptr, acc, fc);
  });
}

// d mu / dx and d var / dx for one slice and one chunk.


// Fixed-order sum of the per-chunk partials, then 1/l_j, the -2 of d var and the discrete mask:
//   dmu[j][c] = invl_j * sum_p gm_part[p][j][c] ;  dvar[j][c] = -2 invl_j * sum_p gv_part[p][j][c]
struct GradReduceParams {
  const double *gm_part, *gv_part;
  int P, d, chunk_ld, count;
  const double *invl;
  unsigned long long disc_bits;
  double *dmu, *dvar;  // [d][chunk_ld] each (this slice's section)
};
__global__ void __launch_bounds__(256) grad_reduce_kernel(GradReduceParams p) {
  const int c = blockIdx.x * 256 + threadIdx.x, j = blockIdx.y;
  if (c >= p.count) return;
  const size_t o0 = (size_t)j * p.chunk_ld + c, st = (size_t)p.d * p.chunk_ld;
  const double am = ordered_sum(p.gm_part + o0, st, p.P), av = ordered_sum(p.gv_part + o0, st, p.P);
  const bool disc = (p.disc_bits >> j) & 1ull;
  const double il = p.invl[j];
  p.dmu[(size_t)j * p.chunk_ld + c] = disc ? 0.0 : am * il;
  p.dvar[(size_t)j * p.chunk_ld + c] = disc ? 0.0 : -2.0 * av * il;
}

// MC-EI adjoint weights (DESIGN.md 2.11): for one eps column e with improvement > 0 at y = mu + sd .* e,
//   A_i += g_i(y),  B_i += g_i(y) e_i,   g_i = df/dy_i of the branch mix_fitness took:
//   affine c_i;  quadratic c_i + 2 q_i (y_i - t_i);  max / min c_i* for the first extreme output i*, 0 for the others
__device__ __forceinline__ void mix_adjoint(const MixParams &mx, const double *y, const double *e, int y_dim, double *A,
                                            double *B) {
  if (mx.kind == 1 || mx.kind == 2) {
    for (int i = 0; i < y_dim; ++i) {
      const double g = mx.kind == 1 ? mx.c[i] : fma(2.0 * mx.q[i], y[i] - mx.t[i], mx.c[i]);
      A[i] += g;
      B[i] = fma(g, e[i], B[i]);
    }
    return;
  }
  int is = -1;   // the selection of mix_fitness: the first output whose term is extreme (NaN terms never reach here)
  double ext = 0.0;
  for (int i = 0; i < y_dim; ++i) {
    if (mx.c[i] == 0.0) continue;
    const double v = fma(mx.c[i], y[i], mx.t[i]);
    if (is < 0 || (mx.kind == 3 ? v > ext : v < ext)) {
      ext = v;
      is = i;
    }
  }
  if (is < 0) return;   // no output enters f: a constant
  A[is] += mx.c[is];
  B[is] = fma(mx.c[is], e[is], B[is]);
}

// Chain rule through EI x PoF.  dmu / dvar: [(sample*y_dim + slice)][d][chunk_ld].
struct AcqGradParams {
  AcqParams a;
  const double *dmu, *dvar;
  const double *prior_mean_grad;  // y_dim x d x M (column-major: index ((m)*d + j)*y_dim + i) or null
  double *grad;                   // d x M, indexed by (m - out_off)
};

// MC = false: the closed-form EI of a LinFitness.  MC = true: the Monte-Carlo EI of a MixParams expression (launched
// only with `best` set; PoF alone has no Monte-Carlo term and takes MC = false).  Per posterior s with eps columns K_s:
//   d EI_s = sum_i A_i d mu_i + B_i d sd_i ,  d sd_i = d var_i / (2 sd_i)  (0 when sd_i == 0 or the variance was clipped)
// with A, B of mix_adjoint averaged over K_s: K_s * y_dim work per posterior, then d * y_dim per candidate.
// Conventions at the measure-zero kinks: the derivative of the branch the value took (imp == 0 contributes 0, a max /
// min tie goes to the first output); a NaN improvement makes the gradient NaN.
template <bool MC>
__global__ void __launch_bounds__(128) acq_grad_kernel(AcqGradParams q) {
  const AcqParams &p = q.a;
  const int c = blockIdx.x * 128 + threadIdx.x;
  const long long m = p.m0 + c;
  if (c >= p.chunk || m >= p.M) return;
  const int d = p.d;
  double gacc[32];
  for (int j = 0; j < d; ++j) gacc[j] = 0.0;
  bool failed = false;
  for (int s = 0; s < p.n_samples; ++s) {
    // pass 1: scalars
    double cdf_i[MAX_YDIM], wmu_i[MAX_YDIM], wvar_i[MAX_YDIM];
    double mu_i[MAX_YDIM], sd_i[MAX_YDIM];   // MC only
    bool live_i[MAX_YDIM];
    double mu_f = 0.0, s2 = 0.0, pof = 1.0;
    for (int i = 0; i < p.y_dim; ++i) {
      const size_t row = (size_t)(s * p.y_dim + i) * p.chunk_ld + c;
      double mu = p.mu[row];
      if (p.prior_mean) mu = p.prior_mean[(size_t)(m - p.in_off) * p.y_dim + i] + mu;
      double var = p.a2[s * p.y_dim + i] - p.sumsq[row] + VAR_JITTER;
      const bool unclipped = var >= 0.0;
      if (!clip_var(var)) failed = true;
      live_i[i] = unclipped;   // the clipped branch of _clip_var returns a constant zero -> zero derivative
      if constexpr (MC) {
        mu_i[i] = mu;
        sd_i[i] = sqrt(var);
      } else {
        mu_f = fma(p.coefs[i], mu, mu_f);
        s2 = fma(p.coefs[i] * p.coefs[i], var, s2);
      }
      cdf_i[i] = 1.0;
      wmu_i[i] = wvar_i[i] = 0.0;
      if (p.has_ymax && !(p.y_max[i] == INFINITY)) {
        const double sd = sqrt(var);
        double z = (p.y_max[i] - mu) / sd;
        if (sd == 0.0 && p.y_max[i] == mu) z = INFINITY;
        cdf_i[i] = norm_cdf(z);
        if (sd > 0.0) {   // d cdf = pdf(z) * ( -dmu/sd - (ymax-mu) dvar / (2 sd var) )
          const double pz = norm_pdf(z);
          wmu_i[i] = -pz / sd;
          wvar_i[i] = -pz * (p.y_max[i] - mu) / (2.0 * sd * var);
        }
        pof *= cdf_i[i];
      }
    }
    double ei = 0.0, cphi = 0.0, cpdf_over_2sf = 0.0;   // d ei = cphi * d mu_f + cpdf_over_2sf * d s2
    double wa[MAX_YDIM], wb[MAX_YDIM];                   // MC: d ei = sum_i wa_i d mu_i + wb_i d var_i
    if constexpr (MC) {
      // the value's loop of acq_candidate (same columns, same order), plus the adjoint weights
      const int k0 = p.n_samples > 1 ? s : 0, k1 = p.n_samples > 1 ? s + 1 : p.mix.n_eps;
      for (int i = 0; i < p.y_dim; ++i) wa[i] = wb[i] = 0.0;
      double tot = 0.0;
      for (int k = k0; k < k1; ++k) {
        double ys[MAX_YDIM];
        const double *ek = p.mix.eps + (size_t)k * p.y_dim;
        for (int i = 0; i < p.y_dim; ++i) ys[i] = mu_i[i] + sd_i[i] * ek[i];
        const double imp = mix_fitness(p.mix, ys, p.y_dim) - p.best;
        tot += (imp != imp) ? imp : (imp > 0.0 ? imp : 0.0);
        if (imp > 0.0) {
          mix_adjoint(p.mix, ys, ek, p.y_dim, wa, wb);
        } else if (imp != imp) {
          for (int i = 0; i < p.y_dim; ++i) wa[i] = wb[i] = NAN;
        }
      }
      const double nk = (double)(k1 - k0);
      ei = tot / nk;
      for (int i = 0; i < p.y_dim; ++i) {
        wa[i] /= nk;
        wb[i] = sd_i[i] > 0.0 ? wb[i] / nk / (2.0 * sd_i[i]) : 0.0;   // a NaN improvement already made wa NaN
      }
    } else if (p.has_best) {
      const double sf = sqrt(s2), diff = mu_f - p.best;
      if (diff == 0.0 && sf == 0.0) {
        ei = 0.0;
      } else {
        const double z = diff / sf;
        const double cz = norm_cdf(z), pz = norm_pdf(z);
        ei = diff * cz + sf * pz;
        if (sf > 0.0) {
          cphi = cz;
          cpdf_over_2sf = pz / (2.0 * sf);
        } else {
          cphi = diff > 0.0 ? 1.0 : 0.0;
        }
      }
    }
    // pass 2: per input dimension
    for (int j = 0; j < d; ++j) {
      double dmu_f = 0.0, ds2 = 0.0, dpof = 0.0, dei_mc = 0.0;
      for (int i = 0; i < p.y_dim; ++i) {
        const size_t row = ((size_t)(s * p.y_dim + i) * d + j) * p.chunk_ld + c;
        double dm = q.dmu[row];
        if (q.prior_mean_grad) dm += q.prior_mean_grad[((size_t)(m - p.in_off) * d + j) * p.y_dim + i];
        const double dv = live_i[i] ? q.dvar[row] : 0.0;
        if constexpr (MC) {
          dei_mc = fma(wa[i], dm, dei_mc);
          dei_mc = fma(wb[i], dv, dei_mc);
        } else {
          dmu_f = fma(p.coefs[i], dm, dmu_f);
          ds2 = fma(p.coefs[i] * p.coefs[i], dv, ds2);
        }
        if (p.has_ymax && !(p.y_max[i] == INFINITY)) {
          double others = 1.0;
          for (int b = 0; b < p.y_dim; ++b)
            if (b != i) others *= cdf_i[b];
          dpof = fma(wmu_i[i] * dm + wvar_i[i] * dv, others, dpof);
        }
      }
      const double dei = MC ? dei_mc : cphi * dmu_f + cpdf_over_2sf * ds2;
      double g;
      if (p.has_best)
        g = p.has_ymax ? dei * pof + ei * dpof : dei;
      else
        g = p.has_ymax ? dpof : 0.0;
      gacc[j] += g;
    }
  }
  bool zero = failed;
  if (p.lb) {
    for (int i = 0; i < d; ++i) {
      const double x = p.Xs[(size_t)(m - p.in_off) * d + i];
      if (x < p.lb[i] || x > p.ub[i]) zero = true;
    }
  }
  if (p.cons_mask && p.cons_mask[m - p.in_off] == 0) zero = true;
  for (int j = 0; j < d; ++j) q.grad[(size_t)(m - p.out_off) * d + j] = zero ? 0.0 : gacc[j] / (double)p.n_samples;
}

// boss_gp_predict_grad's output stage (in place of acq_kernel + acq_grad_kernel): the P = n_samples * y_dim posteriors
// of the chunk, from [q][chunk_ld] rows and [q][j][chunk_ld] sections to the caller's candidate-major layout
//   mu / var / status  at (m - out_off) * P + q ,   dmu / dvar  at ((m - out_off) * d + j) * P + q .
// One thread per output element in output order, so every store is coalesced; the strided loads hit the chunk's
// sections, which the reductions just wrote.  mu and var use acq_candidate's expressions (same bits as boss_gp_predict).
struct PredictGradParams {
  AcqParams a;                     // mu / sumsq rows, a2, prior_mean, any_fail, chunk geometry
  const double *dmu, *dvar;        // [q][d][chunk_ld]
  const double *prior_mean_grad;   // y_dim x d x M (index ((m - in_off) * d + j) * y_dim + i) or null
  double *mu_out, *var_out, *dmu_out, *dvar_out;   // each may be null
  int *status_out;
};
__global__ void __launch_bounds__(256) predict_grad_kernel(PredictGradParams q) {
  const AcqParams &p = q.a;
  const int P = p.n_samples * p.y_dim, d = p.d;
  const int e = blockIdx.x * 256 + threadIdx.x;   // element of the chunk's dmu / dvar output (chunk * d * P < 2^31)
  if (e >= p.chunk * d * P) return;
  const int qi = e % P, j = e / P % d, c = e / (P * d);
  const int i = qi % p.y_dim;
  const size_t row = (size_t)qi * p.chunk_ld + c;
  const long long m = p.m0 + c;
  const double var_raw = p.a2[qi] - p.sumsq[row] + VAR_JITTER;
  const size_t sec = ((size_t)qi * d + j) * p.chunk_ld + c;
  const size_t o = (size_t)(m - p.out_off) * d * P + ((size_t)j * P + qi);   // == ((m - out_off) * d + j) * P + q
  if (q.dmu_out) {
    double dm = q.dmu[sec];
    if (q.prior_mean_grad) dm += q.prior_mean_grad[((size_t)(m - p.in_off) * d + j) * p.y_dim + i];
    q.dmu_out[o] = dm;
  }
  if (q.dvar_out) q.dvar_out[o] = var_raw >= 0.0 ? q.dvar[sec] : 0.0;   // the clipped branch of _clip_var is a constant
  // the first chunk * P threads also write the value outputs, element e of those (candidate-major as well)
  if (e >= p.chunk * P) return;
  const int q2 = e % P, c2 = e / P;
  const size_t row2 = (size_t)q2 * p.chunk_ld + c2;
  const long long m2 = p.m0 + c2;
  double mu = p.mu[row2];
  if (p.prior_mean) mu = p.prior_mean[(size_t)(m2 - p.in_off) * p.y_dim + q2 % p.y_dim] + mu;
  double var = p.a2[q2] - p.sumsq[row2] + VAR_JITTER;
  const bool ok = clip_var(var);
  if (!ok) *p.any_fail = 1;
  const size_t o2 = (size_t)(m2 - p.out_off) * P + q2;
  if (q.mu_out) q.mu_out[o2] = mu;
  if (q.var_out) q.var_out[o2] = var;
  if (q.status_out) q.status_out[o2] = ok ? 0 : 2;
}

}  // namespace boss
