"""ExpectedImprovement acquisition (mirror of src/acquisitions/expected_improvement.jl and src/acquisition.jl).
The closure returned by construct_acquisition evaluates whole candidate matrices in one library call."""
from __future__ import annotations

from dataclasses import dataclass, field

import math

import numpy as np

from . import _lib
from .posterior import model_posterior
from .types import BossOptions, BossProblem, ExprFitness, LinFitness, cons_mask

_erfc = np.vectorize(math.erfc, otypes=[np.float64])


def _normal_cdf(mu, sigma, x):
    """cdf(Normal(mu, sigma), x) as Distributions.jl/StatsFuns evaluate it (erfc form; sigma == 0 with x == mu -> 1;
    an infinite bound -> exactly 1, src/utils/inf.jl:13-15)."""
    with np.errstate(divide="ignore", invalid="ignore"):
        z = (x - mu) / sigma
    z = np.where((sigma == 0.0) & (x == mu), np.inf, z)
    return np.where(np.isposinf(x), 1.0, _erfc(-z * 0.7071067811865476) / 2.0)


def julia_argmax(v):
    """Julia's argmax on a vector: first maximal element under isless (NaN is maximal, -0.0 < +0.0)."""
    v = np.asarray(v, dtype=np.float64)
    nan = np.flatnonzero(np.isnan(v))
    if nan.size:
        return int(nan[0])
    cand = np.flatnonzero(v == v.max())
    if v[cand[0]] == 0.0:
        pos = cand[~np.signbit(v[cand])]
        if pos.size:
            return int(pos[0])
    return int(cand[0])


def julia_sortperm_rev(v):
    """Julia's stable sortperm(v; rev=true): descending under isless (NaN first, +0.0 before -0.0), ties to the lower
    index.  The order of boss_ei_score_topk; its first element is julia_argmax(v)."""
    v = np.asarray(v, dtype=np.float64)
    u = np.ascontiguousarray(v).view(np.uint64)
    key = np.where((u >> np.uint64(63)) != 0, ~u, u | np.uint64(1 << 63))
    key = np.where(np.isnan(v), np.uint64(0xFFFFFFFFFFFFFFFF), key)
    return np.argsort(~key, kind="stable")


def sample_eps(y_dim: int, count: int, rng=None):
    """sample_ϵs (expected_improvement.jl:118): y_dim x count standard normal draws."""
    rng = np.random.default_rng() if rng is None else rng
    return rng.standard_normal((y_dim, count))


@dataclass
class ExpectedImprovement:
    fitness: object
    eps_samples: int = 200
    cons_safe: bool = True


def best_so_far(problem: BossProblem, fitness):
    """expected_improvement.jl:135-140 (raw observations; feasible = all(y .<= y_max))."""
    Y = problem.data.Y
    if Y.size == 0:
        return None
    feas = np.all(Y <= problem.y_max[:, None], axis=0)
    if not feas.any():
        return None
    return float(max(fitness(Y[:, i]) for i in np.flatnonzero(feas)))


class Acquisition:
    """The safe acquisition closure of construct_safe_acquisition (src/acquisition.jl:21-25):
    acq(x::Vector) -> Real, acq(X::Matrix) -> Vector; -inf where the reference's SafeFunction catches an error,
    0. outside the domain (make_safe, expected_improvement.jl:58-65)."""

    def __init__(self, problem: BossProblem, posteriors, ei: ExpectedImprovement, best, eps=None):
        self.problem = problem
        self.posts = posteriors if isinstance(posteriors, list) else [posteriors]
        self.y_dim = problem.data.y_dim
        self.slices = [s.gp for p in self.posts for s in p.slices]
        self.models = [s.model for s in self.posts[0].slices]
        # LinFitness: closed-form EI fused on the device.  NonlinFitness (an arbitrary host closure): the posterior
        # mean / variance of every output come from the device, the Monte-Carlo average over eps
        # (expected_improvement.jl:104-111) is finished on the host.
        self.fitness = ei.fitness
        self.nonlin = not isinstance(ei.fitness, LinFitness)
        self.expr = ei.fitness if isinstance(ei.fitness, ExprFitness) else None    # device MC-EI (boss_mcei_score)
        if self.nonlin:
            count = ei.eps_samples if len(self.posts) == 1 else len(self.posts)   # ϵ_sample_count, :115-116
            self.eps = sample_eps(self.y_dim, count) if eps is None else np.asarray(eps, dtype=np.float64)
            assert self.eps.shape == (self.y_dim, count), (self.eps.shape, (self.y_dim, count))
        self.coefs = None if self.nonlin else np.asarray(ei.fitness.coefs, dtype=np.float64)
        self.best = best
        self.y_max = None if np.all(np.isinf(problem.y_max)) else problem.y_max
        self.cons_safe = ei.cons_safe

    def device_resident_ok(self):
        """True when nothing on the scoring path is a host closure (prior means, `cons`), i.e. the device-resident
        multi-start driver can run the whole solve."""
        probe = np.zeros((self.problem.data.x_dim, 1))
        no_mean = all(m.mean_at(i, probe) is None for i, m in enumerate(self.models))
        return (no_mean and self.problem.domain.cons is None and self.cons_safe
                and (not self.nonlin or self.expr is not None))

    def _fitness_values(self, pred):
        """fitness.(pred_samples): pred is y_dim x P.  A closure written with numpy broadcasting is applied to the
        whole matrix at once; otherwise (scalar-only closure) column by column, as the reference does."""
        P = pred.shape[1]
        try:
            v = np.asarray(self.fitness(pred), dtype=np.float64)
            if v.shape == (P,):
                return v
        except Exception:
            pass
        return np.array([float(self.fitness(pred[:, k])) for k in range(P)])

    def _mc_acq(self, X, want_argmax=False):
        """construct_ei for a NonlinFitness (expected_improvement.jl:68-90, :104-111)."""
        M = X.shape[1]
        if self.expr is not None:     # expression-set fitness: the whole Monte-Carlo EI runs on the device
            lb, ub, cm = self._guards(X)
            e = self.expr
            acq, bv, bi = _lib.mcei_score(self.slices, self.y_dim, len(self.posts), X, e.kind_id, self.eps, self.best,
                                          self.y_max, c0=e.c0, c=e.c, q=e.q, t=e.t, lb=lb, ub=ub, cons_mask=cm,
                                          prior_mean_s=self._prior_mean(X), want_acq=not want_argmax)
            return (int(bi), float(bv)) if want_argmax else acq
        pm = self._prior_mean(X)
        acc = np.zeros(M)
        failed = np.zeros(M, dtype=bool)
        for s, post in enumerate(self.posts):
            mu = np.empty((self.y_dim, M))
            var = np.empty((self.y_dim, M))
            for i, sl in enumerate(post.slices):
                mu[i], var[i], st = _lib.gp_predict(sl.gp, X, None if pm is None else pm[i])
                failed |= st != 0
            if self.best is None and self.y_max is None:
                continue
            with np.errstate(invalid="ignore"):
                sd = np.sqrt(var)
            pof = 1.0 if self.y_max is None else np.prod(_normal_cdf(mu, sd, self.y_max[:, None]), axis=0)
            if self.best is None:
                acc += pof
                continue
            eps = self.eps if len(self.posts) == 1 else self.eps[:, s:s + 1]
            K = eps.shape[1]
            pred = mu[:, :, None] + sd[:, :, None] * eps[:, None, :]                      # y_dim x M x K
            f = self._fitness_values(pred.reshape(self.y_dim, M * K)).reshape(M, K)
            acc += np.maximum(0.0, f - self.best).sum(axis=1) / K * pof
        acq = np.where(failed, -np.inf, acc / len(self.posts))
        lb, ub, cm = self._guards(X)
        if lb is not None:
            acq = np.where(np.all((X >= np.asarray(lb)[:, None]) & (X <= np.asarray(ub)[:, None]), axis=0), acq, 0.0)
        if cm is not None:
            acq = np.where(np.asarray(cm, dtype=bool), acq, 0.0)
        return acq

    def _prior_mean(self, X):
        ms = [m.mean_at(i, X) for i, m in enumerate(self.models)]
        if all(v is None for v in ms):
            return None
        return np.stack([np.zeros(X.shape[1]) if v is None else v for v in ms])

    def _guards(self, X):
        if not self.cons_safe:
            return None, None, None
        lb, ub = self.problem.domain.bounds
        return lb, ub, cons_mask(X, self.problem.domain)

    def __call__(self, x):
        x = np.asarray(x, dtype=np.float64)
        vec = x.ndim == 1
        X = x[:, None] if vec else x
        if self.nonlin:
            acq = self._mc_acq(X)
            return float(acq[0]) if vec else acq
        lb, ub, cm = self._guards(X)
        acq, _, _ = _lib.ei_score(self.slices, self.y_dim, len(self.posts), X, self.coefs, self.best, self.y_max,
                                  lb, ub, cm, self._prior_mean(X))
        return float(acq[0]) if vec else acq

    def argmax(self, X):
        """-> (index, value) with Julia argmax semantics, one fused launch sequence (no score vector round trip)."""
        X = np.asarray(X, dtype=np.float64)
        if self.nonlin:
            if self.expr is not None:
                return self._mc_acq(X, want_argmax=True)
            acq = self._mc_acq(X)
            bi = julia_argmax(acq)
            return int(bi), float(acq[bi])
        lb, ub, cm = self._guards(X)
        _, bv, bi = _lib.ei_score(self.slices, self.y_dim, len(self.posts), X, self.coefs, self.best, self.y_max,
                                  lb, ub, cm, self._prior_mean(X), want_acq=False)
        return int(bi), float(bv)

    def topk(self, X, k):
        """-> (indices (k,), values (k,)) of the k best columns of X in julia_sortperm_rev order.  LinFitness and
        ExprFitness select on the device (boss_ei_score_topk, boss_mcei_score_topk); an opaque NonlinFitness scores
        every column and sorts on the host."""
        X = np.asarray(X, dtype=np.float64)
        if self.expr is not None:
            lb, ub, cm = self._guards(X)
            e = self.expr
            vals, idx = _lib.mcei_score_topk(self.slices, self.y_dim, len(self.posts), X, e.kind_id, self.eps, self.best,
                                             self.y_max, k, c0=e.c0, c=e.c, q=e.q, t=e.t, lb=lb, ub=ub, cons_mask=cm,
                                             prior_mean_s=self._prior_mean(X))
            return idx, vals
        if self.nonlin:
            acq = self._mc_acq(X)
            top = julia_sortperm_rev(acq)[:k]
            return top, acq[top]
        lb, ub, cm = self._guards(X)
        vals, idx = _lib.ei_score_topk(self.slices, self.y_dim, len(self.posts), X, self.coefs, self.best, self.y_max, k,
                                       lb, ub, cm, self._prior_mean(X))
        return idx, vals

    def value_and_grad(self, X):
        """-> acq (M,), grad (d, M).  Prior-mean gradients are not propagated for closure means."""
        X = np.asarray(X, dtype=np.float64)
        if self.expr is not None:     # expression-set fitness: the chain rule through the Monte-Carlo EI on the device
            lb, ub, cm = self._guards(X)
            e = self.expr
            return _lib.mcei_value_grad(self.slices, self.y_dim, len(self.posts), X, e.kind_id, self.eps, self.best,
                                        self.y_max, c0=e.c0, c=e.c, q=e.q, t=e.t, lb=lb, ub=ub, cons_mask=cm,
                                        prior_mean_s=self._prior_mean(X))
        if self.nonlin:
            raise NotImplementedError("NonlinFitness: the Monte-Carlo EI of an arbitrary host closure has no analytic "
                                      "gradient here (the reference pushes ForwardDiff duals through the closure); "
                                      "use GridAM / SamplingAM / RandomAM or a derivative-free OptimizationAM")
        lb, ub, cm = self._guards(X)
        return _lib.ei_value_grad(self.slices, self.y_dim, len(self.posts), X, self.coefs, self.best, self.y_max,
                                  lb, ub, cm, self._prior_mean(X))


def construct_acquisition(problem: BossProblem, options: BossOptions = BossOptions(), eps=None) -> Acquisition:
    """construct_acquisition(::ExpectedImprovement, problem, options) (expected_improvement.jl:49-56).
    Refits the posterior exactly like the reference (model_posterior on every call)."""
    ei = problem.acquisition
    post = model_posterior(problem)
    b = best_so_far(problem, ei.fitness)
    if options.info and b is None:
        print("Warning: No feasible solution in the dataset yet. Cannot calculate EI!")
    return Acquisition(problem, post, ei, b, eps)


construct_safe_acquisition = construct_acquisition
