// acq.cuh -- the acquisition value of one candidate from its posterior means (and variances): closed-form or
// Monte-Carlo EI x PoF with the guards.  Used by acq_kernel and the fused epilogues in score.cuh, and by the FP32 mean
// tier's bound kernel in tk_score.cu.
#pragma once
#include "kernel_fn.cuh"

namespace boss {

constexpr int MAX_YDIM = 16;

// Monte-Carlo expected improvement for a NonlinFitness drawn from a small expression set
// (expected_improvement(::NonlinFitness, ...), src/acquisitions/expected_improvement.jl:104-111):
//   EI = 1/K sum_k max(0, f(mu + sqrt(var) .* eps_k) - best),   f one of
//   kind 1  affine     f(y) = c0 + sum_i c_i y_i
//   kind 2  quadratic  f(y) = c0 + sum_i c_i y_i + sum_i q_i (y_i - t_i)^2
//   kind 3  max        f(y) = c0 + max_i (c_i y_i + t_i)   over the outputs with c_i != 0
//   kind 4  min        f(y) = c0 + min_i (c_i y_i + t_i)   over the outputs with c_i != 0
// kind 0 = off (LinFitness closed form).  An arbitrary Julia closure stays a host job (INTEGRATION.md).
constexpr int MIX_MAX_EPS = 4096;
struct MixParams {
  int kind = 0, n_eps = 0;
  double c0 = 0.0;
  double c[MAX_YDIM] = {}, q[MAX_YDIM] = {}, t[MAX_YDIM] = {};
  const double *eps = nullptr;        // device, y_dim x n_eps column-major
  const double *eps_host = nullptr;   // host copy handed in by the caller (uploaded by score_core)
};
__host__ __device__ __forceinline__ double mix_fitness(const MixParams &mx, const double *y, int y_dim) {
  double f = mx.c0;
  if (mx.kind == 1) {
    for (int i = 0; i < y_dim; ++i) f = fma(mx.c[i], y[i], f);
  } else if (mx.kind == 2) {
    for (int i = 0; i < y_dim; ++i) {
      const double dv = y[i] - mx.t[i];
      f = fma(mx.c[i], y[i], f);
      f = fma(mx.q[i] * dv, dv, f);
    }
  } else {
    bool any = false;
    double ext = 0.0;
    for (int i = 0; i < y_dim; ++i) {
      if (mx.c[i] == 0.0) continue;
      const double v = fma(mx.c[i], y[i], mx.t[i]);
      if (!any) {
        ext = v;
        any = true;
      } else if (v != v || ext != ext) {
        ext = NAN;
      } else {
        ext = mx.kind == 3 ? (v > ext ? v : ext) : (v < ext ? v : ext);
      }
    }
    f += ext;
  }
  return f;
}

struct AcqParams {
  int y_dim, n_samples, d;
  long long M, m0;       // global candidate count / chunk start
  long long in_off;      // Xs / prior_mean / cons_mask are indexed by (m - in_off)
  long long out_off;     // acq / mu_out / var_out / status_out are indexed by (m - out_off)
  int chunk;             // candidates in this chunk
  int chunk_ld;          // leading dimension of mu / sumsq ([n_samples*y_dim][chunk_ld])
  const double *mu;      // K*^T alpha per (sample, slice)
  const double *sumsq;   // |W k*|^2 per (sample, slice)
  const double *a2;      // [n_samples*y_dim] prior variance a^2 (device)
  const double *prior_mean;  // y_dim x M or null
  double coefs[MAX_YDIM];
  double y_max[MAX_YDIM];
  int has_best, has_ymax;
  double best;
  const double *Xs;      // d x M for the bounds check (null if no bounds)
  const double *lb, *ub; // device, d each (null if no bounds)
  const unsigned char *cons_mask;  // or null
  double *acq;           // or null
  double *mu_out, *var_out;  // predict mode (single slice) or null
  int *status_out;       // predict mode or null
  int *any_fail;         // device flag
  double *blk_val;       // per-block winners
  long long *blk_idx;
  MixParams mix;         // kind != 0: Monte-Carlo EI of a NonlinFitness expression instead of the closed form
};

__device__ __forceinline__ double norm_cdf(double z) { return 0.5 * erfc(-z * 0.7071067811865476); }
__device__ __forceinline__ double norm_pdf(double z) { return exp(-0.5 * z * z) * 0.3989422804014327; }


// The acquisition value of candidate c of the chunk (global index m): slices x BI samples -> EI x PoF, guards.
// Writes the optional per-candidate outputs.  Shared by acq_kernel and the fused epilogues of score_trmm_kernel and
// screen_mean_bound_kernel.  The candidate's mean of slice q is mu_c[q * mu_ld].  BOUND: the bound pass of argmax
// screening, whose parameters have no sumsq, PoF, Monte-Carlo term, guards or per-candidate outputs other than acq; the
// compiler then drops those branches (and their registers) from the same arithmetic.
template <bool BOUND = false>
__device__ __forceinline__ double acq_candidate(const AcqParams &p, const int c, const long long m, const double *mu_c,
                                                size_t mu_ld) {
  double result;
  {
    const bool has_ymax = !BOUND && p.has_ymax, mixed = !BOUND && p.mix.kind != 0;
    const double *sumsq = BOUND ? nullptr : p.sumsq;
    double accum = 0.0;
    bool failed = false;
    for (int s = 0; s < p.n_samples; ++s) {
      double mu_f = 0.0, s2 = 0.0, pof = 1.0;
      double mu_i[MAX_YDIM], sd_i[MAX_YDIM];
      for (int i = 0; i < p.y_dim; ++i) {
        const size_t row = (size_t)(s * p.y_dim + i) * p.chunk_ld + c;
        double mu = mu_c[(size_t)(s * p.y_dim + i) * mu_ld];
        if (p.prior_mean) mu = p.prior_mean[(size_t)(m - p.in_off) * p.y_dim + i] + mu;
        // sumsq == null: the prior variance a^2 + 1e-18, an upper bound of the posterior one (argmax screening)
        double var = p.a2[s * p.y_dim + i] - (sumsq ? sumsq[row] : 0.0) + VAR_JITTER;
        const bool ok = clip_var(var);
        if (!ok) failed = true;
        if (!BOUND && p.mu_out) p.mu_out[m - p.out_off] = mu;
        if (!BOUND && p.var_out) p.var_out[m - p.out_off] = var;
        if (!BOUND && p.status_out) p.status_out[m - p.out_off] = ok ? 0 : 2;
        mu_f = fma(p.coefs[i], mu, mu_f);
        s2 = fma(p.coefs[i] * p.coefs[i], var, s2);
        mu_i[i] = mu;
        sd_i[i] = sqrt(var);
        if (has_ymax) {
          const double ym = p.y_max[i];
          if (!(ym == INFINITY)) {                 // cdf(., Infinity()) == 1 exactly (src/utils/inf.jl:13-15)
            const double sd = sqrt(var);
            double z = (ym - mu) / sd;
            if (sd == 0.0 && ym == mu) z = INFINITY;   // StatsFuns: x == mu, sigma == 0 -> cdf 1
            pof *= norm_cdf(z);
          }
        }
      }
      double a;
      if (p.has_best && mixed) {
        // one posterior: all eps columns; BI posteriors: posterior s takes column s (expected_improvement.jl:87-90,108-111)
        const int k0 = p.n_samples > 1 ? s : 0, k1 = p.n_samples > 1 ? s + 1 : p.mix.n_eps;
        double tot = 0.0;
        for (int k = k0; k < k1; ++k) {
          double ys[MAX_YDIM];
          for (int i = 0; i < p.y_dim; ++i) ys[i] = mu_i[i] + sd_i[i] * p.mix.eps[(size_t)k * p.y_dim + i];
          const double imp = mix_fitness(p.mix, ys, p.y_dim) - p.best;
          tot += (imp != imp) ? imp : (imp > 0.0 ? imp : 0.0);   // max(0, NaN) = NaN in Julia
        }
        const double ei = tot / (double)(k1 - k0);
        a = has_ymax ? ei * pof : ei;
      } else if (p.has_best) {
        const double sf = sqrt(s2);
        const double diff = mu_f - p.best;
        double ei;
        if (diff == 0.0 && sf == 0.0) {
          ei = 0.0;
        } else {
          const double z = diff / sf;
          ei = diff * norm_cdf(z) + sf * norm_pdf(z);
        }
        a = has_ymax ? ei * pof : ei;
      } else {
        a = has_ymax ? pof : 0.0;
      }
      accum += a;
    }
    result = accum / (double)p.n_samples;
    if (failed) {
      result = -INFINITY;
      *p.any_fail = 1;
    }
    if (!BOUND && p.lb) {
      bool inb = true;
      for (int i = 0; i < p.d; ++i) {
        const double x = p.Xs[(size_t)(m - p.in_off) * p.d + i];
        if (x < p.lb[i] || x > p.ub[i]) inb = false;
      }
      if (!inb) result = 0.0;
    }
    if (!BOUND && p.cons_mask && p.cons_mask[m - p.in_off] == 0) result = 0.0;
    if (p.acq) p.acq[m - p.out_off] = result;
  }
  return result;
}
__device__ __forceinline__ double acq_candidate(const AcqParams &p, const int c, const long long m) {
  return acq_candidate(p, c, m, p.mu + c, (size_t)p.chunk_ld);
}

}  // namespace boss
