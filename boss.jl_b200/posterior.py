"""model_posterior dispatch (mirror of src/posterior.jl): problem -> params -> slices, broadcast over BI samples."""
from __future__ import annotations

import numpy as np

from . import _lib
from .gaussian_process import GaussianProcessPosterior, _as_gp, _kernel_parts, _raise_domain_error, model_posterior_slice
from .types import BossProblem, get_params


class DefaultModelPosterior:
    """src/posterior.jl:31-79: stacks y_dim independent slices."""

    def __init__(self, slices):
        self.slices = slices

    def mean_and_var(self, x):
        res = [s.mean_and_var(x) for s in self.slices]
        x = np.asarray(x)
        if x.ndim == 1:
            return np.array([r[0] for r in res]), np.array([r[1] for r in res])
        return np.stack([r[0] for r in res]), np.stack([r[1] for r in res])      # y_dim x M

    def mean_and_var_grad(self, x):
        """mean_and_var with the x-gradients of every output slice in one boss_gp_predict_grad call (the mirror's
        stand-in for ForwardDiff through mean_and_var): vector x -> (mu (y_dim,), var (y_dim,), dmu (y_dim, d),
        dvar (y_dim, d)); matrix X (d x M) -> (mu (y_dim, M), var (y_dim, M), dmu (y_dim, d, M), dvar (y_dim, d, M)).
        Prior-mean closures are not differentiated.  Raises ValueError where mean_and_var does."""
        x = np.asarray(x, dtype=np.float64)
        vec = x.ndim == 1
        X = x[:, None] if vec else x
        ms = [s.model.mean_at(s.slice_idx, X) for s in self.slices]
        pm = None if all(m is None for m in ms) else np.stack([np.zeros(X.shape[1]) if m is None else m for m in ms])
        mu, var, dmu, dvar, st = _lib.gp_predict_grad([s.gp for s in self.slices], len(self.slices), 1, X, pm)
        _raise_domain_error(var, st)
        if vec:
            return mu[:, 0].copy(), var[:, 0].copy(), dmu[:, :, 0].copy(), dvar[:, :, 0].copy()
        return mu, var, dmu, dvar

    def mean(self, x):
        return self.mean_and_var(x)[0]

    def var(self, x):
        return self.mean_and_var(x)[1]

    def std(self, x):
        return np.sqrt(self.var(x))

    def mean_and_std(self, x):
        mu, var = self.mean_and_var(x)
        return mu, np.sqrt(var)

    def mean_and_cov(self, X):
        """src/posterior.jl:73-78: (mu (y_dim, M), Sigma (M, M, y_dim))"""
        res = [s.mean_and_cov(X) for s in self.slices]
        return np.stack([r[0] for r in res]), np.stack([r[1] for r in res], axis=2)

    def cov(self, X):
        """src/posterior.jl:55-57"""
        return self.mean_and_cov(X)[1]


def model_posterior(problem_or_model, params=None, data=None):
    """model_posterior(problem) | model_posterior(model, params, data); a list of params (BIParams)
    broadcasts to a list of posteriors (src/posterior.jl:15-16)."""
    if isinstance(problem_or_model, BossProblem):
        prob = problem_or_model
        return model_posterior(prob.model, get_params(prob.params), prob.data)
    model = problem_or_model
    params = get_params(params)
    if isinstance(params, (list, tuple)):
        return _model_posterior_batch(model, list(params), data)
    return DefaultModelPosterior([model_posterior_slice(model, params, data, i) for i in range(data.y_dim)])


def _model_posterior_batch(model, plist, data):
    """BI samples (src/posterior.jl:15-16 broadcasts model_posterior over the samples, one Cholesky each): here all
    samples of one output slice are factored by ONE boss_gp_fit_batch call."""
    S = len(plist)
    gms = [_as_gp(model, p) for p in plist]
    kid, mask = _kernel_parts(gms[0][0].kernel)
    slices = [[None] * data.y_dim for _ in range(S)]
    for i in range(data.y_dim):
        means = [gm.mean_at(i, data.X) for gm, _ in gms]
        Ymm = np.stack([data.Y[i] - (0.0 if m is None else m) for m in means])
        L = np.stack([gp.lengthscales[:, i] for _, gp in gms])
        A = np.array([gp.amplitudes[i] for _, gp in gms])
        N = np.array([gp.noise_std[i] for _, gp in gms])
        handles = _lib.gp_fit_batch(data.X, Ymm, L, A, N, kid, mask)
        for s, h in enumerate(handles):
            if h is None:
                raise ValueError("PosDefException: kernel matrix is not positive definite")
            slices[s][i] = GaussianProcessPosterior(h, gms[s][0], i)
    return [DefaultModelPosterior(sl) for sl in slices]


def average_mean(posteriors, x):
    """src/posterior.jl:177-179"""
    return sum(p.mean(x) for p in posteriors) / len(posteriors)
