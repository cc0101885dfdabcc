"""Model fitters that build log-likelihood batches (mirror of src/model_fitters/sampling.jl, optimization.jl)."""
from __future__ import annotations

from typing import Optional

import numpy as np

from .gaussian_process import (GaussianProcessParams, Semiparametric, SemiparametricParams, data_loglike,
                               data_loglike_and_grad)
from .types import BossOptions, BossProblem, MAPParams


class SamplingMAP:
    """sampling.jl:8-78: draw `samples` prior samples, keep the one with the highest model log-likelihood
    (strict `v > best_v`, i.e. first maximum) -- evaluated as ONE batch."""

    def __init__(self, samples: int = 200, seed: Optional[int] = None):
        self.samples = samples
        self.rng = np.random.default_rng(seed)


class OptimizationMAP:
    """optimization.jl:23-164.  All multistarts advance together and every evaluation of all of them is one batched
    device call.  algorithm:
      "lbfgs"    gradient-based (the reference's default autodiff = AutoForwardDiff(), optimization.jl:41,153): batched
                 L-BFGS in log-parameter space on boss_gp_loglik_grad_batch (value + analytic gradient of the data
                 log-likelihood for all starts at once; the prior term's gradient is a host-side central difference).
                 GaussianProcess models, and Semiparametric models whose Parametric has a `jacobian` (theta enters raw,
                 its gradient from boss_gp_loglik_grad_batch_mean); a Semiparametric model without one falls back to
                 "compass".
      "compass"  derivative-free compass search in log space (what NEWUOA / BOBYQA are used for in the examples)."""

    def __init__(self, multistart=20, iters: int = 40, step0: float = 0.5, seed: Optional[int] = None,
                 algorithm: str = "lbfgs"):
        self.multistart = multistart          # an int, or a list of start params (SampleOptMAP hands its best samples over)
        self.iters = iters
        self.step0 = step0
        self.algorithm = algorithm
        self.rng = np.random.default_rng(seed)


class SampleOptMAP:
    """sample_opt.jl:37-48: SamplingMAP (return_all) -> the `multistart` best samples -> OptimizationMAP from them."""

    def __init__(self, samples: int = 200, multistart: int = 20, iters: int = 40, seed: Optional[int] = None,
                 algorithm: str = "lbfgs"):
        self.samples = samples
        self.multistart = multistart
        self.iters = iters
        self.algorithm = algorithm
        self.rng = np.random.default_rng(seed)


def model_loglike(model, data):
    """model_loglike = data_loglike + params_loglike (src/types/surrogate_model.jl:135-142); accepts a list."""
    dll = data_loglike(model, data)
    pll = model.params_loglike()

    def ll(params):
        if isinstance(params, (list, tuple)):
            prior = np.array([pll(p) for p in params])
            ok = np.isfinite(prior)
            out = np.full(len(params), -np.inf)
            if ok.any():
                out[ok] = dll([p for p, k in zip(params, ok) if k]) + prior[ok]
            return out
        pr = pll(params)
        return -np.inf if not np.isfinite(pr) else dll(params) + pr
    return ll


def _dirac_mask(model, template):
    """True for parameters pinned by a Dirac prior: they are excluded from the search vector, like the reference's
    create_dirac_mask / filter_diracs (src/models/utils/dirac.jl, gaussian_process.jl:300-328)."""
    from .types import Dirac, Product
    gp = model.nonparametric if isinstance(model, Semiparametric) else model
    mask = []
    if isinstance(template, SemiparametricParams):
        mask += [isinstance(pr, Dirac) for pr in model.parametric.theta_priors]
    for pr in gp.lengthscale_priors:                       # column-major vec(lambda): slice by slice
        parts = pr.parts if isinstance(pr, Product) else [pr] * template.lengthscales.shape[0]
        mask += [isinstance(q, Dirac) for q in parts]
    mask += [isinstance(pr, Dirac) for pr in gp.amplitude_priors]
    mask += [isinstance(pr, Dirac) for pr in gp.noise_std_priors]
    return np.array(mask, dtype=bool)


def _vectorize(p):
    parts = [np.log(p.lengthscales.ravel(order="F")), np.log(p.amplitudes), np.log(p.noise_std)]
    if isinstance(p, SemiparametricParams):
        parts.insert(0, p.theta)
    return np.concatenate(parts)


def _offsets(template):
    k = template.theta.shape[0] if isinstance(template, SemiparametricParams) else 0
    nl = template.lengthscales.size
    na = template.amplitudes.shape[0]
    return {"lengthscales": slice(k, k + nl), "amplitudes": slice(k + nl, k + nl + na),
            "noise_std": slice(k + nl + na, None)}


def _devectorize(template, v):
    k = 0
    theta = None
    if isinstance(template, SemiparametricParams):
        k = template.theta.shape[0]
        theta = v[:k]
    shp = template.lengthscales.shape
    nl = shp[0] * shp[1]
    lam = np.exp(v[k:k + nl]).reshape(shp, order="F")
    na = template.amplitudes.shape[0]
    amp = np.exp(v[k + nl:k + nl + na])
    ns = np.exp(v[k + nl + na:])
    if theta is not None:
        return SemiparametricParams(theta.copy(), lam, amp, ns)
    return GaussianProcessParams(lam, amp, ns)


def estimate_parameters(fitter, problem: BossProblem, options: BossOptions = BossOptions(), return_all: bool = False):
    model, data = problem.model, problem.data
    ll = model_loglike(model, data)
    sampler = model.params_sampler(fitter.rng)
    if isinstance(fitter, SamplingMAP):
        samples = [sampler() for _ in range(fitter.samples)]
        vals = ll(samples)
        if return_all:
            return [MAPParams(p, float(v)) for p, v in zip(samples, vals)]
        b = int(np.argmax(vals))                       # first maximum == the reference's strict `v > best_v`
        return MAPParams(samples[b], float(vals[b]))
    if isinstance(fitter, SampleOptMAP):
        # sample_opt.jl:41-46: all samples with their log-likelihoods, sorted, the best `multistart` become the starts
        sm = SamplingMAP(fitter.samples)
        sm.rng = fitter.rng
        allp = estimate_parameters(sm, problem, options, return_all=True)
        order = np.argsort([-p.loglike for p in allp], kind="stable")[: fitter.multistart]
        om = OptimizationMAP([allp[i].params for i in order], fitter.iters, algorithm=fitter.algorithm)
        om.rng = fitter.rng
        return estimate_parameters(om, problem, options, return_all=return_all)
    if isinstance(fitter, OptimizationMAP):
        starts = list(fitter.multistart) if not isinstance(fitter.multistart, int) else [sampler() for _ in range(fitter.multistart)]
        tmpl = starts[0]
        fixed = _dirac_mask(model, tmpl)
        V0 = np.stack([_vectorize(p) for p in starts])             # S x P_all
        free = np.flatnonzero(~fixed)
        exact = [_vectorize(p) for p in starts]

        def _devec_free(s_idx, vfree):
            """Rebuild params from the free sub-vector; Dirac-pinned entries keep their exact sampled value."""
            full = exact[s_idx].copy()
            full[free] = vfree
            p = _devectorize(tmpl, full)
            ref = starts[s_idx]
            for name in ("lengthscales", "amplitudes", "noise_std"):
                a, b = getattr(p, name), getattr(ref, name)
                fm = fixed[_offsets(tmpl)[name]].reshape(b.shape, order="F")
                a[fm] = b[fm]
            return p
        V = V0[:, free]
        S, P = V.shape
        if P == 0:
            f0 = ll(starts)
            b = int(np.argmax(f0))
            return MAPParams(starts[b], float(f0[b]))
        _devectorize_rows = lambda rows, owners: [_devec_free(o, v) for v, o in zip(rows, owners)]
        if fitter.algorithm == "lbfgs" and (not isinstance(model, Semiparametric) or model.parametric.jacobian is not None):
            lo, hi = _search_box(model, V0)
            return _lbfgs_map(fitter, model, data, V, free, tmpl, _devec_free, return_all, lo[free], hi[free])
        f = ll(_devectorize_rows(V, range(S)))
        step = np.full(S, fitter.step0)
        for _ in range(fitter.iters):
            probes = []
            for j in range(P):
                for sgn in (1.0, -1.0):
                    Vp = V.copy(); Vp[:, j] += sgn * step
                    probes.append(Vp)
            allp = np.concatenate(probes)                           # (2P*S) x P
            fv = ll(_devectorize_rows(allp, list(range(S)) * (2 * P))).reshape(2 * P, S)
            best_probe = np.argmax(fv, axis=0)
            fbest = fv[best_probe, np.arange(S)]
            improve = fbest > f
            Vnew = np.stack(probes)[best_probe, np.arange(S)]
            V = np.where(improve[:, None], Vnew, V)
            f = np.where(improve, fbest, f)
            step = np.where(improve, step, step * 0.5)
            if np.all(step < 1e-4):
                break
        if np.all(np.isneginf(f)):
            raise RuntimeError("All optimization runs failed!")
        if return_all:
            return [MAPParams(_devec_free(i, v), float(x)) for i, (v, x) in enumerate(zip(V, f)) if np.isfinite(x)]
        b = int(np.argmax(f))
        return MAPParams(_devec_free(b, V[b]), float(f[b]))
    raise TypeError(f"unsupported model fitter {type(fitter).__name__}")


def _search_box(model, V0):
    """Box of the gradient search over the whole vectorised parameters (_vectorize order), from the starts V0 (S x P_all).
    batched_lbfgs_maximize needs a finite box, and its first trial step is a tenth of the widest side.  The log-parameters
    get [-30, 30] (e^30: effectively unbounded).  theta enters raw, on a scale only the starts reveal: it gets
    [min over starts - 30, max over starts + 30], cut to the support of a Uniform prior (outside it the prior term is
    -inf).  Its sides are 60 + the spread of the starts in that entry, so starts spread wider than a few units (a wide
    Normal prior) enlarge the first trial step of every entry, log-parameters included; the Armijo backtracking then
    halves the step until it is accepted, at the cost of extra evaluations in the first rounds."""
    from .types import Uniform
    lo = np.full(V0.shape[1], -30.0)
    hi = np.full(V0.shape[1], 30.0)
    if isinstance(model, Semiparametric):
        k = len(model.parametric.theta_priors)
        lo[:k] = V0[:, :k].min(axis=0) - 30.0
        hi[:k] = V0[:, :k].max(axis=0) + 30.0
        for c, pr in enumerate(model.parametric.theta_priors):
            if isinstance(pr, Uniform):
                lo[c], hi[c] = max(lo[c], pr.lo), min(hi[c], pr.hi)
    return lo, hi


def _lbfgs_map(fitter, model, data, V, free, tmpl, devec_free, return_all, lo, hi):
    """Gradient OptimizationMAP: maximise data_loglike + params_loglike over the free parameters of all starts (log
    scale for lambda, alpha, sigma; raw theta) inside the box [lo, hi] with the batched L-BFGS of
    acquisition_maximizers.batched_lbfgs_maximize.  One value + gradient evaluation of all unfinished starts = one
    boss_gp_loglik_grad_batch (Semiparametric: boss_gp_loglik_grad_batch_mean) call per output slice."""
    from .acquisition_maximizers import batched_lbfgs_maximize
    llg = data_loglike_and_grad(model, data)
    pll = model.params_loglike()
    S, P = V.shape
    off = _offsets(tmpl)
    owners = {"n": 0}

    def prior_and_grad(p, vfree, s_idx):
        base = pll(p)
        g = np.zeros(P)
        if not np.isfinite(base):
            return base, g
        h = 1e-6
        for k in range(P):                       # O(#params) host work per start: central difference of the prior term
            vp, vm = vfree.copy(), vfree.copy()
            vp[k] += h; vm[k] -= h
            fp, fm = pll(devec_free(s_idx, vp)), pll(devec_free(s_idx, vm))
            g[k] = (fp - fm) / (2 * h) if np.isfinite(fp) and np.isfinite(fm) else 0.0
        return base, g

    def value_and_grad(Z):                      # Z: P x m (columns = the unfinished starts, in the order given by `act`)
        cols = value_and_grad.active
        plist = [devec_free(s, Z[:, c]) for c, s in enumerate(cols)]
        ll_d, grads = llg(plist)
        f = np.empty(len(cols)); G = np.zeros((P, len(cols)))
        for c, (s, p) in enumerate(zip(cols, plist)):
            parts = [grads[c].lengthscales.ravel(order="F") * p.lengthscales.ravel(order="F"),
                     grads[c].amplitudes * p.amplitudes, grads[c].noise_std * p.noise_std]          # d/d log(lambda, alpha, sigma)
            if isinstance(p, SemiparametricParams):
                parts.insert(0, grads[c].theta)                                                     # theta is not log-scaled
            full = np.concatenate(parts)
            pr, gpr = prior_and_grad(p, Z[:, c], s)
            f[c] = ll_d[c] + pr if np.isfinite(pr) else -np.inf
            G[:, c] = full[free] + gpr
        return f, G

    # batched_lbfgs_maximize calls value_and_grad on the columns of the unfinished starts; it needs to know which
    # starts those are (Dirac-pinned entries are rebuilt per start), so the driver publishes the active set
    X, f = batched_lbfgs_maximize(value_and_grad, V.T.copy(), lo, hi, iters=fitter.iters, publish_active=value_and_grad)
    if np.all(np.isneginf(f)):
        raise RuntimeError("All optimization runs failed!")
    if return_all:
        return [MAPParams(devec_free(i, X[:, i]), float(f[i])) for i in range(S) if np.isfinite(f[i])]
    b = int(np.argmax(f))
    return MAPParams(devec_free(b, X[:, b]), float(f[b]))
