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


def _pof_grad(mu, var, sd, dmu, dvar, y_max):
    """d PoF / dx for one posterior: PoF = prod_i cdf(Normal(mu_i, sd_i), y_max_i), by the product rule over the outputs;
    d cdf_i = pdf(z_i) (-d mu_i / sd_i - (y_max_i - mu_i) d var_i / (2 sd_i var_i)), 0 where sd_i == 0 or y_max_i = +Inf.
    mu, var, sd (y_dim, M); dmu, dvar (y_dim, d, M) -> (d, M)."""
    ym = np.asarray(y_max, dtype=np.float64)[:, None]
    cdf = _normal_cdf(mu, sd, ym)
    with np.errstate(divide="ignore", invalid="ignore"):
        z = (ym - mu) / sd
        pdf = np.exp(-0.5 * z * z) * 0.3989422804014327
        dc = pdf[:, None, :] * (-dmu / sd[:, None, :] - (ym - mu)[:, None, :] * dvar / (2.0 * sd * var)[:, None, :])
    dc = np.where(((sd > 0.0) & ~np.isposinf(ym))[:, None, :], dc, 0.0)
    dpof = np.zeros(dmu.shape[1:])
    for i in range(mu.shape[0]):
        others = np.prod(np.delete(cdf, i, axis=0), axis=0)
        dpof += dc[i] * others
    return dpof


def mc_ei_value_grad(mu, var, dmu, dvar, eps, f, g, best, y_max, status=None):
    """Value and x-gradient of the Monte-Carlo EI (x PoF) of a NonlinFitness closure (expected_improvement.jl:104-111)
    from the posteriors and their x-gradients, by the chain rule of DESIGN.md 2.11 with g = df/dy taken from the caller:
      y_k = mu + sd .* eps_k,  imp_k = f(y_k) - best,  EI_s = 1/K sum_k max(0, imp_k)
      d EI_s = sum_i A_i d mu_i + B_i d sd_i,  A_i = 1/K sum_{imp_k > 0} g_i(y_k),  B_i = 1/K sum_{imp_k > 0} g_i(y_k) eps_ik
    d sd_i = d var_i / (2 sd_i) where sd_i > 0 (dvar is already 0 where the variance was clipped); a NaN improvement gives
    a NaN gradient; PoF enters by the product rule; the BI samples are averaged.
      mu, var (S, y_dim, M); dmu, dvar (S, y_dim, d, M); eps (y_dim, K) (S > 1: posterior s takes column s);
      f(Y) -> (P,), g(Y) -> (y_dim, P) for Y (y_dim, P); best / y_max None or as Acquisition; status (S, y_dim, M) or None.
    -> val (M,) (-inf where a status is non-zero; bit for bit Acquisition's value path), grad (d, M) (0 there).
    No domain guards."""
    S, y_dim, M = mu.shape
    d = dmu.shape[2]
    acc = np.zeros(M)
    gacc = np.zeros((d, M))
    failed = np.zeros(M, dtype=bool) if status is None else np.any(np.asarray(status) != 0, axis=(0, 1))
    for s in range(S):
        m, v, dm, dv = mu[s], var[s], dmu[s], dvar[s]
        if best is None and y_max is None:
            continue
        with np.errstate(invalid="ignore"):
            sd = np.sqrt(v)
        # the value: the expressions of Acquisition._mc_acq, so the bits agree
        pof = 1.0 if y_max is None else np.prod(_normal_cdf(m, sd, y_max[:, None]), axis=0)
        dpof = 0.0 if y_max is None else _pof_grad(m, v, sd, dm, dv, y_max)
        if best is None:
            acc += pof
            gacc += dpof
            continue
        e = eps if S == 1 else eps[:, s:s + 1]
        K = e.shape[1]
        pred = (m[:, :, None] + sd[:, :, None] * e[:, None, :]).reshape(y_dim, M * K)      # y_dim x M x K
        imp = f(pred).reshape(M, K) - best
        ei = np.maximum(0.0, imp).sum(axis=1) / K
        acc += ei * pof
        pos = (imp > 0.0)[None]
        G = np.where(pos, np.asarray(g(pred), dtype=np.float64).reshape(y_dim, M, K), 0.0)
        A = G.sum(axis=2) / K
        B = (G * e[:, None, :]).sum(axis=2) / K
        A = np.where(np.isnan(imp).any(axis=1)[None], np.nan, A)
        with np.errstate(divide="ignore", invalid="ignore"):
            dsd = np.where(sd[:, None, :] > 0, dv / (2.0 * sd[:, None, :]), 0.0)
        dei = np.einsum("im,idm->dm", A, dm) + np.einsum("im,idm->dm", B, dsd)
        gacc += dei if y_max is None else dei * pof + ei * dpof
    val = np.where(failed, -np.inf, acc / S)
    grad = np.where(failed[None], 0.0, gacc / S)
    return val, grad


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

    def _fitness_grads(self, pred):
        """fitness.grad at the columns of pred (y_dim x P) -> y_dim x P; column by column for a closure that does not
        broadcast, like _fitness_values."""
        P = pred.shape[1]
        g = self.fitness.grad
        try:
            v = np.asarray(g(pred), dtype=np.float64)
            if v.shape == (self.y_dim, P):
                return v
        except Exception:
            pass
        return np.stack([np.asarray(g(pred[:, k]), dtype=np.float64).reshape(self.y_dim) for k in range(P)], axis=1)

    def _apply_guards(self, X, acq, grad=None):
        """make_safe (expected_improvement.jl:58-65): 0 outside the bounds or `cons` (the gradient too)."""
        lb, ub, cm = self._guards(X)
        keep = np.ones(X.shape[1], dtype=bool)
        if lb is not None:
            keep &= np.all((X >= np.asarray(lb)[:, None]) & (X <= np.asarray(ub)[:, None]), axis=0)
        if cm is not None:
            keep &= np.asarray(cm, dtype=bool)
        acq = np.where(keep, acq, 0.0)
        return acq if grad is None else (acq, np.where(keep[None], grad, 0.0))

    def _mc_value_grad(self, X):
        """Value and x-gradient of the Monte-Carlo EI of a NonlinFitness closure with `grad`: the posteriors and their
        x-gradients of all S*y_dim slices in one boss_gp_predict_grad call, the chain rule on the host
        (mc_ei_value_grad).  The value equals acq(X) bit for bit."""
        S, M, d = len(self.posts), X.shape[1], X.shape[0]
        mu, var, dmu, dvar, st = _lib.gp_predict_grad(self.slices, self.y_dim, S, X, self._prior_mean(X))
        acq, grad = mc_ei_value_grad(mu.reshape(S, self.y_dim, M), var.reshape(S, self.y_dim, M),
                                     dmu.reshape(S, self.y_dim, d, M), dvar.reshape(S, self.y_dim, d, M), self.eps,
                                     self._fitness_values, self._fitness_grads, self.best, self.y_max,
                                     status=st.reshape(S, self.y_dim, M))
        return self._apply_guards(X, acq, grad)

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
        return self._apply_guards(X, acq)

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
        """-> acq (M,), grad (d, M).  Prior-mean gradients are not propagated for closure means.  A NonlinFitness needs
        `grad` (df/dy) unless it is an ExprFitness."""
        X = np.asarray(X, dtype=np.float64)
        if self.expr is not None:     # expression-set fitness: the chain rule through the Monte-Carlo EI on the device
            lb, ub, cm = self._guards(X)
            e = self.expr
            return _lib.mcei_value_grad(self.slices, self.y_dim, len(self.posts), X, e.kind_id, self.eps, self.best,
                                        self.y_max, c0=e.c0, c=e.c, q=e.q, t=e.t, lb=lb, ub=ub, cons_mask=cm,
                                        prior_mean_s=self._prior_mean(X))
        if self.nonlin and getattr(self.fitness, "grad", None) is not None:
            return self._mc_value_grad(X)       # a closure with df/dy: the chain rule on the host
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
