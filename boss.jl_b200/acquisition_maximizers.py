"""Acquisition maximizers that build candidate batches (mirror of src/acquisition_maximizers/*.jl).
Each one turns the reference's per-point loop into one batched scoring call."""
from __future__ import annotations

import itertools
from dataclasses import dataclass
from typing import Optional

import numpy as np

import copy

from . import _lib
from .acquisition import Acquisition, best_so_far, construct_safe_acquisition
from .posterior import average_mean, model_posterior
from .types import BossOptions, BossProblem, Domain, ExperimentData, discrete_round, generate_LHC, in_domain


class GridAM:
    """grid.jl:24-65.  `points` are generated once from the domain, filtered by in_domain."""

    def __init__(self, problem: BossProblem, steps, shuffle: bool = True, seed: Optional[int] = None):
        dom = problem.domain
        lb, ub = dom.bounds
        ranges = []
        for lo, hi, st, disc in zip(lb, ub, steps, dom.discrete):
            if disc:
                st = float(np.ceil(st))
                ranges.append(np.arange(np.ceil(lo), np.floor(hi) + 0.5 * st, st))
            else:
                cnt = int(np.floor((hi - lo) / st + 1e-12)) + 1
                ranges.append(lo + st * np.arange(cnt))
        # Iterators.product: first dimension varies fastest
        pts = [np.array(p[::-1]) for p in itertools.product(*ranges[::-1])]
        self.points = np.array([p for p in pts if in_domain(p, dom)]).T          # d x M
        self.steps = steps
        self.shuffle = shuffle
        self.rng = np.random.default_rng(seed)


class SamplingAM:
    """sampling.jl:8-57: draw `samples` points from x_prior restricted to the domain, score, argmax."""

    def __init__(self, x_prior, samples: int, max_attempts: int = 200, seed: Optional[int] = None):
        self.x_prior = x_prior            # callable rng -> x (d,), or None = uniform over the bounds
        self.samples = samples
        self.max_attempts = max_attempts
        self.rng = np.random.default_rng(seed)


class OptimizationAM:
    """optimization.jl:20-118: multi-start local optimisation.  Here all starts advance in lock-step: every
    iteration is ONE batched value+gradient call (projected L-BFGS with backtracking)."""

    def __init__(self, multistart=200, iters: int = 60, history: int = 8, seed: Optional[int] = None):
        self.multistart = multistart
        self.iters = iters
        self.history = history
        self.rng = np.random.default_rng(seed)


class SampleOptAM:
    """sample_opt.jl:41-52: SamplingAM (return_all) -> best `multistart` samples -> OptimizationAM from them."""

    def __init__(self, x_prior, samples: int, multistart: int, iters: int = 60, seed: Optional[int] = None):
        self.sampler = SamplingAM(x_prior, samples, seed=seed)
        self.multistart = multistart
        self.iters = iters


class SequentialBatchAM:
    """batch.jl:1-38: pick `batch_size` candidates sequentially, extending the data set after each pick with the
    speculative point (x, posterior mean at x).  The reference refits every GP from scratch per pick
    (`model_posterior(problem)` in speculative_evaluation!); here the fitted factor caches are extended in place
    with one O(n^2) boss_gp_append per slice (hyper-parameters do not change between picks)."""

    def __init__(self, am, batch_size: int):
        self.am = am
        self.batch_size = batch_size


def _rand_in_domain(am: SamplingAM, domain: Domain):
    lb, ub = domain.bounds
    for _ in range(am.max_attempts):
        x = am.x_prior(am.rng) if am.x_prior is not None else am.rng.uniform(lb, ub)
        x = discrete_round(domain.discrete, x)
        if in_domain(x, domain):
            return x
    return None


def _draw_samples(am: SamplingAM, domain: Domain):
    """sampling.jl:37-48: `samples` rejection-sampled points (d x M); the ones that failed are dropped."""
    xs = [x for x in (_rand_in_domain(am, domain) for _ in range(am.samples)) if x is not None]
    if not xs:
        raise RuntimeError("SamplingAM: No samples were successfully drawn!")
    return np.stack(xs, axis=1)


def batched_lbfgs_maximize(value_and_grad, starts, lb, ub, iters=60, history=8, discrete=None, publish_active=None):
    """Maximise f over the box [lb, ub] from every column of `starts` simultaneously (projected L-BFGS with Armijo
    backtracking).  value_and_grad(X: d x S) -> (f: S, g: d x S).  Returns X (d x S), f (S).

    Host twin of the device-resident driver (csrc/multistart.cuh, boss_ei_maximize_multistart): every start is its own
    state machine - own history ring, own step counter, own termination - and one ROUND advances every unfinished
    start by exactly one function evaluation (all their trial points in one batched call).  A start is finished after
    `iters` accepted steps, when an accepted step no longer moves it, or when 12 step sizes in a row were rejected along
    the projected gradient (after 12 rejections along an L-BFGS direction the history is dropped first)."""
    X = np.clip(np.array(starts, dtype=np.float64, copy=True), lb[:, None], ub[:, None])
    d, S = X.shape
    if publish_active is not None:           # callers whose closure needs to know which starts a batch belongs to
        publish_active.active = np.arange(S)
    f, g = value_and_grad(X)
    f = np.where(np.isfinite(f), f, -np.inf)
    g = np.array(g, dtype=np.float64, copy=True)
    H = max(1, min(history, 15))
    Sh = np.zeros((H, d, S)); Yh = np.zeros((H, d, S))       # per-start rings, oldest first in rows [0, hist_len)
    hist_len = np.zeros(S, dtype=int)
    state = np.zeros(S, dtype=int) if iters > 0 else np.full(S, 2)          # 0 needs a direction, 1 line search, 2 finished
    steps = np.zeros(S, dtype=int); trials = np.zeros(S, dtype=int)
    t = np.ones(S); dirn = np.zeros((d, S))
    step0 = 0.1 * np.max(ub - lb)
    for _ in range(2 * iters + 12 if iters > 0 else 0):
        act = np.flatnonzero(state != 2)
        if act.size == 0:
            break
        for m in np.flatnonzero(state == 0):                  # two-loop recursion on the start's own history
            bound = ((X[:, m] <= lb) & (g[:, m] < 0)) | ((X[:, m] >= ub) & (g[:, m] > 0))
            pg = np.where(bound, 0.0, g[:, m])                 # projected gradient
            q = pg.copy()
            hl = hist_len[m]
            al, rh = np.zeros(hl), np.zeros(hl)
            for k in range(hl - 1, -1, -1):
                rh[k] = 1.0 / max(Sh[k, :, m] @ Yh[k, :, m], 1e-300)
                al[k] = rh[k] * (Sh[k, :, m] @ q)
                q -= al[k] * Yh[k, :, m]
            sd = step0 / max(np.linalg.norm(pg), 1e-300)
            if hl > 0:
                gamma = (Sh[hl - 1, :, m] @ Yh[hl - 1, :, m]) / max(Yh[hl - 1, :, m] @ Yh[hl - 1, :, m], 1e-300)
                q *= gamma if (np.isfinite(gamma) and gamma > 0) else 1.0
            else:
                q *= sd
            for k in range(hl):
                q += Sh[k, :, m] * (al[k] - rh[k] * (Yh[k, :, m] @ q))
            q[bound] = 0.0                                     # stay on the active bounds
            dirn[:, m] = q if (q @ pg) > 0 else pg * sd        # not an ascent direction -> projected steepest ascent
            t[m] = 1.0; trials[m] = 0; state[m] = 1
        Xt = np.clip(X[:, act] + dirn[:, act] * t[act], lb[:, None], ub[:, None])
        if publish_active is not None:
            publish_active.active = act
        ft, gt = value_and_grad(Xt)
        ft = np.where(np.isfinite(ft), ft, -np.inf)
        for c, m in enumerate(act):
            if ft[c] >= f[m] + 1e-4 * (g[:, m] @ (Xt[:, c] - X[:, m])):
                sk, yk = Xt[:, c] - X[:, m], -(gt[:, c] - g[:, m])          # curvature pair for maximisation
                if sk @ yk > 1e-16:
                    if hist_len[m] == H:
                        Sh[:-1, :, m] = Sh[1:, :, m]; Yh[:-1, :, m] = Yh[1:, :, m]
                        hist_len[m] -= 1
                    Sh[hist_len[m], :, m] = sk; Yh[hist_len[m], :, m] = yk
                    hist_len[m] += 1
                moved = np.max(np.abs(sk))
                X[:, m], f[m], g[:, m] = Xt[:, c], ft[c], gt[:, c]
                steps[m] += 1
                state[m] = 2 if (steps[m] >= iters or moved < 1e-10) else 0
            else:
                t[m] *= 0.5
                trials[m] += 1
                state[m] = 1
                if trials[m] >= 12:        # drop the history and retry along the projected gradient; finished if that fails too
                    state[m] = 0 if hist_len[m] > 0 else 2
                    hist_len[m] = 0
    return X, f


def _sequential_batch(sb: SequentialBatchAM, problem: BossProblem, options: BossOptions):
    prob = copy.copy(problem)                                       # deepcopy(problem) of batch.jl:27 (data only)
    prob.data = ExperimentData(problem.data.X.copy(), problem.data.Y.copy())
    posts = model_posterior(prob)                                   # ONE fit; extended in place below
    post_list = posts if isinstance(posts, list) else [posts]
    picks = []
    for _ in range(sb.batch_size):
        acq = Acquisition(prob, posts, prob.acquisition, best_so_far(prob, prob.acquisition.fitness))
        x, _ = maximize_acquisition(sb.am, prob, options, acq=acq)
        y = average_mean(post_list, x) if len(post_list) > 1 else post_list[0].mean(x)     # batch.jl:35
        prob.data.augment(x, y)
        for p in post_list:
            for i, sl in enumerate(p.slices):
                m = sl.model.mean_at(i, x[:, None])
                if not _lib.gp_append(sl.gp, x, y[i] - (0.0 if m is None else float(m[0]))):
                    raise ValueError("PosDefException: kernel matrix is not positive definite")
        picks.append(x)
    return np.stack(picks, axis=1), None


def maximize_acquisition(am, problem: BossProblem, options: BossOptions = BossOptions(), return_all: bool = False,
                         acq=None):
    """-> (x, val).  src/types/acquisition_maximizer.jl:12-20.  `acq`: reuse an already constructed acquisition."""
    if isinstance(am, SequentialBatchAM):
        return _sequential_batch(am, problem, options)
    if acq is None:
        acq = construct_safe_acquisition(problem, options)
    dom = problem.domain
    if isinstance(am, GridAM):
        pts = am.points[:, am.rng.permutation(am.points.shape[1])] if am.shuffle else am.points   # grid.jl:47
        idx, val = acq.argmax(pts)
        return pts[:, idx].copy(), val
    if isinstance(am, SamplingAM):
        X = _draw_samples(am, dom)
        if return_all:
            return X, acq(X)
        idx, val = acq.argmax(X)
        return X[:, idx].copy(), val
    if isinstance(am, SampleOptAM):
        # the `multistart` best samples, selected on the device (Acquisition.topk: isless order, NaN first)
        X = _draw_samples(am.sampler, dom)
        top, _ = acq.topk(X, min(am.multistart, X.shape[1]))
        return maximize_acquisition(OptimizationAM(X[:, top], am.iters), problem, options, acq=acq)
    if isinstance(am, OptimizationAM):
        lb, ub = dom.bounds
        if isinstance(am.multistart, int):
            starts = (0.5 * (lb + ub))[:, None] if am.multistart == 1 else generate_LHC(dom.bounds, am.multistart, am.rng)
        else:
            starts = np.asarray(am.multistart, dtype=np.float64)
        if acq.device_resident_ok():
            # no host closures on the path (prior mean, cons): the whole multi-start solve stays on the device
            dm = dom.discrete if dom.discrete.any() else None
            if acq.expr is not None:
                e = acq.expr
                _, f, bx, bv, _, _ = _lib.mcei_maximize_multistart(acq.slices, acq.y_dim, len(acq.posts), starts, e.kind_id,
                                                                   acq.eps, acq.best, acq.y_max, lb, ub, c0=e.c0, c=e.c,
                                                                   q=e.q, t=e.t, iters=am.iters, history=am.history,
                                                                   discrete_mask=dm)
            else:
                _, f, bx, bv, _, _ = _lib.ei_maximize_multistart(acq.slices, acq.y_dim, len(acq.posts), starts, acq.coefs,
                                                                 acq.best, acq.y_max, lb, ub, am.iters, am.history,
                                                                 discrete_mask=dm)
            if np.isneginf(bv):
                raise RuntimeError("All optimization runs failed!")                  # optim_multistart.jl:34
            return bx, bv
        X, f = batched_lbfgs_maximize(acq.value_and_grad, starts, lb, ub, am.iters, am.history)
        if np.all(np.isneginf(f)):
            raise RuntimeError("All optimization runs failed!")                      # optim_multistart.jl:34
        b = int(np.argmax(f))                                                         # first maximal
        x = discrete_round(dom.discrete, X[:, b])                                     # optimization.jl:116
        return x, acq(x)
    raise TypeError(f"unsupported acquisition maximizer {type(am).__name__}")
