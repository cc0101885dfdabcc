// multistart.cuh -- per-start pieces of the device-resident multi-start optimiser (projected L-BFGS with Armijo
// backtracking, maximisation).  One thread per start.
//
// Reference: OptimizationAM (src/acquisition_maximizers/optimization.jl:55-118) runs `multistart` independent
// local solves through optimize_multistart (src/utils/optim_multistart.jl:10-90), each evaluating acq(x) one
// point at a time.  Here every start is its own small state machine (needs a direction -> in a line search ->
// finished) and one ROUND advances every unfinished start by exactly one function evaluation: the trial points of
// all unfinished starts are compacted into one batch and scored by one pass of the scoring pipeline (score.cuh /
// grad.cuh) on device-resident points.  A start that has to backtrack simply spends more rounds on that step while
// the others move on, so every evaluation batch is as full as the set of unfinished starts allows (the round-1
// lock-step driver re-evaluated a handful of stragglers up to 12 times per iteration at the full latency of a
// pass over W: 162 passes for 59 batches' worth of work at n = 4096).  No state is shared between starts - history
// ring, step counter and termination are per start - so a start's trajectory does not depend on which other
// starts are in the batch, and therefore not on how the starts are sharded over GPUs.
#pragma once
#include <type_traits>

#include "common.cuh"

namespace boss {

constexpr int MS_MAXD = 32;            // acquisition driver: x_dim <= 32
constexpr int MS_MAP_MAXD = 34;        // hyper-parameter driver (boss_gp_map_multistart): d + 2 <= 34 entries
constexpr int MS_MAXH = 16;
constexpr int MS_MAX_TRIALS = 12;     // step sizes 1, 1/2, ..., 2^-11 per line search

// MAXD: the dimension capacity (per-thread arrays of the two-loop recursion, the box); a driver instantiates the
// kernels below at its own capacity
template <int MAXD>
struct MsStateT {
  int d, H, iters;           // H = ring capacity; iters = accepted steps after which a start is finished
  long long M;
  double *X, *f, *g;         // [M][d], [M], [M][d]  current (accepted) point, value, gradient
  double *Xc, *fc, *gc;      // compact batch of this round: trial points / values / gradients (capacity M)
  double *dirn, *t;          // [M][d], [M] search direction and current step size
  double *Sh, *Yh;           // [H][M][d] curvature pairs, one ring per start
  int *hist_len, *hist_start, *trials, *steps;   // [M] each
  int *nev;                  // [M] evaluations a start has spent (trial points examined); it is cut off at `budget`
  int budget;                // = 2 iters + MS_MAX_TRIALS: a start may reject every other trial on average
  int *state;                // [M] 0 = needs a direction, 1 = in a line search, 2 = finished
  int *idx;                  // [cap] compact list: idx[slot] = start
  int fan;                   // trial points per unfinished start in this round (speculative step-size fan, see below)
  double lb[MAXD], ub[MAXD];
  double step0;
  int *counters;             // [0] length of this round's compact list, [1] starts still unfinished after the round,
                             // [2] running total of the evaluations a one-trial-per-round search would have made
};
using MsState = MsStateT<MS_MAXD>;

__device__ __forceinline__ double ms_clip(double v, double lo, double hi) { return v < lo ? lo : (v > hi ? hi : v); }

template <int MAXD>
__global__ void ms_init_kernel(MsStateT<MAXD> st, const double *starts) {
  const long long m = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (m >= st.M) return;
  for (int j = 0; j < st.d; ++j) st.X[m * st.d + j] = ms_clip(starts[m * st.d + j], st.lb[j], st.ub[j]);
  st.hist_len[m] = st.hist_start[m] = st.trials[m] = st.steps[m] = st.nev[m] = 0;
  st.state[m] = st.iters > 0 ? 0 : 2;
}

// non-finite acquisition values (SafeFunction's -Inf, NaN) count as -Inf
__global__ void ms_sanitize_kernel(double *f, long long M) {
  const long long m = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (m < M && !isfinite(f[m])) f[m] = -INFINITY;
}

// Every unfinished start contributes `fan` trial points to this round's batch: the step sizes t, t/2, ... its
// backtracking search would try one after the other.  fan = 1 is plain one-evaluation-per-round backtracking; once few
// starts are left a pass over W costs the same for 1 or 64 points (it is bound by the length of the DMMA accumulation
// chain), so the next step sizes ride along and a start that has to backtrack does not spend another round on it.  The
// trials are examined in order and the first acceptable one wins, so the trajectory is exactly the sequential one.
// A start that has just accepted a step (or has not moved yet) first gets its L-BFGS ascent direction from its own
// history (two-loop recursion).
template <int MAXD>
__global__ void ms_propose_kernel(MsStateT<MAXD> st) {
  const long long m = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (m >= st.M || st.state[m] == 2) return;
  const int d = st.d;
  if (st.state[m] == 0) {
    const int hist_len = st.hist_len[m], hist_start = st.hist_start[m];
    double q[MAXD], gl[MAXD], al[MS_MAXH], rh[MS_MAXH];
    double gnorm2 = 0.0;
    using Mask = typename std::conditional<(MAXD > 32), unsigned long long, unsigned>::type;
    Mask bound = 0;   // coordinates that sit on a bound with the gradient pointing out of the box
    for (int j = 0; j < d; ++j) {
      const double x = st.X[m * d + j], gj = st.g[m * d + j];
      const bool out = (x <= st.lb[j] && gj < 0.0) || (x >= st.ub[j] && gj > 0.0);
      bound |= out ? (Mask(1) << j) : Mask(0);
      gl[j] = out ? 0.0 : gj;            // projected gradient
      q[j] = gl[j];
      gnorm2 = fma(gl[j], gl[j], gnorm2);
    }
    const double sd = st.step0 / fmax(sqrt(gnorm2), 1e-300);
    for (int k = hist_len - 1; k >= 0; --k) {        // newest -> oldest
      const size_t o = ((size_t)((hist_start + k) % st.H) * st.M + m) * d;
      double sy = 0.0, sq = 0.0;
      for (int j = 0; j < d; ++j) {
        sy = fma(st.Sh[o + j], st.Yh[o + j], sy);
        sq = fma(st.Sh[o + j], q[j], sq);
      }
      rh[k] = 1.0 / fmax(sy, 1e-300);
      al[k] = rh[k] * sq;
      for (int j = 0; j < d; ++j) q[j] = fma(-al[k], st.Yh[o + j], q[j]);
    }
    if (hist_len > 0) {
      const size_t o = ((size_t)((hist_start + hist_len - 1) % st.H) * st.M + m) * d;
      double sy = 0.0, yy = 0.0;
      for (int j = 0; j < d; ++j) {
        sy = fma(st.Sh[o + j], st.Yh[o + j], sy);
        yy = fma(st.Yh[o + j], st.Yh[o + j], yy);
      }
      const double gamma = sy / fmax(yy, 1e-300);
      const double sc = (isfinite(gamma) && gamma > 0.0) ? gamma : 1.0;
      for (int j = 0; j < d; ++j) q[j] *= sc;
    } else {
      for (int j = 0; j < d; ++j) q[j] *= sd;
    }
    for (int k = 0; k < hist_len; ++k) {             // oldest -> newest
      const size_t o = ((size_t)((hist_start + k) % st.H) * st.M + m) * d;
      double yq = 0.0;
      for (int j = 0; j < d; ++j) yq = fma(st.Yh[o + j], q[j], yq);
      const double b = rh[k] * yq;
      for (int j = 0; j < d; ++j) q[j] = fma(st.Sh[o + j], al[k] - b, q[j]);
    }
    double dg = 0.0;
    for (int j = 0; j < d; ++j) {
      if ((bound >> j) & Mask(1)) q[j] = 0.0;             // stay on the active bounds
      dg = fma(q[j], gl[j], dg);
    }
    const bool bad = !(dg > 0.0);                    // not an ascent direction -> steepest ascent
    for (int j = 0; j < d; ++j) st.dirn[m * d + j] = bad ? gl[j] * sd : q[j];
    st.t[m] = 1.0;
    st.trials[m] = 0;
    st.state[m] = 1;
  }
  const int slot0 = atomicAdd(&st.counters[0], st.fan);   // the order of the batch does not matter: scores are per point
  double t = st.t[m];
  for (int k = 0; k < st.fan; ++k, t *= 0.5) {            // slots beyond the start's remaining trials are ignored later
    st.idx[slot0 + k] = (int)m;
    for (int j = 0; j < d; ++j)
      st.Xc[(size_t)(slot0 + k) * d + j] = ms_clip(fma(st.dirn[m * d + j], t, st.X[m * d + j]), st.lb[j], st.ub[j]);
  }
}

// Armijo test of this round's trial points.  Accepted: curvature pair into the start's own ring, move, count the
// step; finished after `iters` steps or when the step no longer moves the point.  Rejected: halve the step; after
// MS_MAX_TRIALS step sizes the history is dropped and the search restarts along the projected gradient, and a start
// whose projected-gradient search fails as well is finished (no acceptable step exists any more).
template <int MAXD>
__global__ void ms_advance_kernel(MsStateT<MAXD> st, int count) {
  const int grp = blockIdx.x * blockDim.x + threadIdx.x;   // one thread per start of the round = per group of `fan` slots
  if (grp >= count) return;
  const long long m = st.idx[grp * st.fan];
  const int d = st.d;
  // trials the sequential search would still make: to the end of this line search, and within the start's budget of
  // evaluations (the budget is per start, not per round, so a trajectory does not depend on the fan width and therefore
  // not on which other starts share the batch)
  const int nk = min(min(st.fan, MS_MAX_TRIALS - st.trials[m]), st.budget - st.nev[m]);
  int state = 1, used = nk;
  for (int k = 0; k < nk; ++k) {
    const size_t slot = (size_t)grp * st.fan + k;
    double ft = st.fc[slot];
    if (!isfinite(ft)) ft = -INFINITY;
    double slope = 0.0;
    for (int j = 0; j < d; ++j) slope = fma(st.g[m * d + j], st.Xc[slot * d + j] - st.X[m * d + j], slope);
    if (ft >= st.f[m] + 1e-4 * slope) {
      double sy = 0.0, mv = 0.0;
      for (int j = 0; j < d; ++j) {
        const double s = st.Xc[slot * d + j] - st.X[m * d + j], y = -(st.gc[slot * d + j] - st.g[m * d + j]);
        sy = fma(s, y, sy);
        mv = fmax(mv, fabs(s));
      }
      if (sy > 1e-16) {   // a safely positive curvature pair: push it (dropping the oldest when the ring is full)
        int hl = st.hist_len[m], hs = st.hist_start[m];
        const int ring = (hs + hl) % st.H;
        const size_t o = ((size_t)ring * st.M + m) * d;
        for (int j = 0; j < d; ++j) {
          st.Sh[o + j] = st.Xc[slot * d + j] - st.X[m * d + j];
          st.Yh[o + j] = -(st.gc[slot * d + j] - st.g[m * d + j]);
        }
        if (hl == st.H - 1)
          hs = (hs + 1) % st.H;
        else
          ++hl;
        st.hist_len[m] = hl;
        st.hist_start[m] = hs;
      }
      for (int j = 0; j < d; ++j) {
        st.X[m * d + j] = st.Xc[slot * d + j];
        st.g[m * d + j] = st.gc[slot * d + j];
      }
      st.f[m] = ft;
      const int steps = ++st.steps[m];
      state = (steps >= st.iters || mv < 1e-10) ? 2 : 0;
      used = k + 1;
      break;
    }
    st.t[m] *= 0.5;
    if (++st.trials[m] >= MS_MAX_TRIALS) {
      // no step size along this direction is acceptable: with curvature history, forget it and retry along the
      // projected gradient; a failed steepest-ascent search means the start cannot improve any more
      state = st.hist_len[m] > 0 ? 0 : 2;
      st.hist_len[m] = 0;
      st.hist_start[m] = 0;
    }
  }
  atomicAdd(&st.counters[2], used);   // evaluations the sequential search would have made (the rest was speculation)
  if ((st.nev[m] += used) >= st.budget) state = 2;   // out of budget: stays at its last accepted point
  st.state[m] = state;
  if (state != 2) atomicAdd(&st.counters[1], 1);
}

// affine prior mean m_i(x) = c_i + b_i . x evaluated on the device (constant means and linear parametric models
// of a Semiparametric surrogate; general closures stay on the host): aff[i*(d+1)] = c_i, aff[i*(d+1)+1+j] = b_ij
__global__ void ms_affine_mean_kernel(const double *X, long long M, int d, int y_dim, const double *aff, double *pm,
                                      double *pmg) {
  const long long m = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (m >= M) return;
  for (int i = 0; i < y_dim; ++i) {
    double v = aff[i * (d + 1)];
    for (int j = 0; j < d; ++j) {
      v = fma(aff[i * (d + 1) + 1 + j], X[m * d + j], v);
      pmg[((size_t)m * d + j) * y_dim + i] = aff[i * (d + 1) + 1 + j];
    }
    pm[(size_t)m * y_dim + i] = v;
  }
}

// final discrete rounding (optimization.jl:116-117)
__global__ void ms_round_kernel(double *X, long long M, int d, unsigned long long disc_bits) {
  const long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (e >= M * d) return;
  if ((disc_bits >> (e % d)) & 1ull) X[e] = rint(X[e]);
}

// ---- hyper-parameter fit (boss_gp_map_multistart, DESIGN.md 2.15) -------------------------------------------------
// A start is one (output slice, start) pair; its P = d + 2 entries [lambda_1..lambda_d, alpha, sigma] are searched in
// z = log(raw).  Prior kinds per entry: 0 Dirac(v) (pinned: raw = v, z stays 0), 1 Normal(mu, s), 2 LogNormal(mu, s),
// 3 Uniform(lo, hi) (inclusive), with the log-densities of boss.jl_b200/types.py.
struct MapEvalParams {
  const double *Z;          // [count][P] points of this batch in z
  const int *idx;           // slot -> local start (the round's compact list), or null: slot k is start k
  long long count;          // slots in the batch
  long long pair0;          // global (slice, start) index of local start 0: slice = (pair0 + start) / M
  long long M;              // starts per slice
  int d, n;
  const int *kind;          // [y_dim][P]
  const double *par;        // [y_dim][P][2]
  const double *Y;          // [y_dim][n] data minus prior mean
  double *ls, *amp, *noise; // [count][d], [count], [count] raw hyper-parameters of the slots
  double *ybuf;             // [count][n] the slot's slice row of Y (null: not gathered)
  const double *ll, *graw;  // log-likelihood and its raw gradient of the slots ([count], [count][P])
  double *f, *g;            // [count], [count][P] value and z-gradient of the slots
};

// one block per slot: raw hyper-parameters (exp(z), or the pinned value) and the slot's Y row
__global__ void map_prep_kernel(MapEvalParams p) {
  const long long k = blockIdx.x;
  const long long m = p.idx ? p.idx[k] : k;
  const int sl = (int)((p.pair0 + m) / p.M), P = p.d + 2;
  for (int j = threadIdx.x; j < P; j += blockDim.x) {
    const int e = sl * P + j;
    const double raw = p.kind[e] == 0 ? p.par[2 * e] : exp(p.Z[k * P + j]);
    if (j < p.d)
      p.ls[k * p.d + j] = raw;
    else if (j == p.d)
      p.amp[k] = raw;
    else
      p.noise[k] = raw;
  }
  if (p.ybuf)
    for (int i = threadIdx.x; i < p.n; i += blockDim.x) p.ybuf[k * p.n + i] = p.Y[(size_t)sl * p.n + i];
}

// one thread per slot: value = log-likelihood + log-prior at the raw values, gradient in z = raw * dll/draw +
// dlogprior/dz (0 for a pinned entry); a non-finite value (K not positive definite, a Uniform support left) is -Inf
// with a zero gradient
__global__ void map_prior_kernel(MapEvalParams p) {
  const long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (k >= p.count) return;
  const long long m = p.idx ? p.idx[k] : k;
  const int sl = (int)((p.pair0 + m) / p.M), P = p.d + 2;
  const double ln_sqrt2pi = 0.91893853320467274178;   // log(sqrt(2 pi))
  double v = p.ll[k];
  for (int j = 0; j < P; ++j) {
    const int e = sl * P + j, kind = p.kind[e];
    double dz = 0.0;
    if (kind != 0) {
      const double x = j < p.d ? p.ls[k * p.d + j] : j == p.d ? p.amp[k] : p.noise[k];
      const double a = p.par[2 * e], b = p.par[2 * e + 1];
      double lp = 0.0, dlp = 0.0;
      if (kind == 1) {          // Normal: -r^2/2 - log(s sqrt(2 pi)), r = (x - mu)/s;  d/dz = x d/dx
        const double r = (x - a) / b;
        lp = -0.5 * r * r - (log(b) + ln_sqrt2pi);
        dlp = -r / b * x;
      } else if (kind == 2) {   // LogNormal: -r^2/2 - log(x s sqrt(2 pi)), r = (log x - mu)/s
        const double r = (log(x) - a) / b;
        lp = -0.5 * r * r - log(x * b * 2.50662827463100050242);
        dlp = -r / b - 1.0;
      } else {                  // Uniform(lo, hi), inclusive
        lp = (a <= x && x <= b) ? -log(b - a) : -INFINITY;
      }
      v += lp;
      dz = fma(x, p.graw[k * P + j], dlp);
    }
    p.g[k * P + j] = dz;
  }
  const bool ok = isfinite(v);
  p.f[k] = ok ? v : -INFINITY;
  if (!ok)
    for (int j = 0; j < P; ++j) p.g[k * P + j] = 0.0;
}

}  // namespace boss
