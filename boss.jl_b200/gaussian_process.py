"""GaussianProcess / Semiparametric surrogate models backed by libboss_b200 (mirror of
src/models/gaussian_process.jl and src/models/semiparametric.jl)."""
from __future__ import annotations

from dataclasses import dataclass
from typing import Callable, List, Optional, Sequence, Union

import numpy as np

from . import _lib
from .types import ExperimentData, Prior


# ---- kernels (KernelFunctions names) -----------------------------------------------------------------
@dataclass(frozen=True)
class SqExponentialKernel:
    kernel_id: int = _lib.KERNEL_SE


@dataclass(frozen=True)
class Matern32Kernel:
    kernel_id: int = _lib.KERNEL_MATERN32


@dataclass(frozen=True)
class Matern52Kernel:
    kernel_id: int = _lib.KERNEL_MATERN52


@dataclass(frozen=True)
class DiscreteKernel:
    """src/models/utils/kernels.jl:43-69: round the flagged dims before evaluating the kernel."""
    kernel: object
    dims: tuple

    @property
    def kernel_id(self):
        return self.kernel.kernel_id


def _kernel_parts(kernel):
    if isinstance(kernel, DiscreteKernel):
        return kernel.kernel_id, np.asarray(kernel.dims, dtype=np.uint8)
    return kernel.kernel_id, None


@dataclass
class GaussianProcessParams:
    """GaussianProcessParams(λ, α, σ): λ is x_dim x y_dim (gaussian_process.jl:58-60)."""
    lengthscales: np.ndarray
    amplitudes: np.ndarray
    noise_std: np.ndarray


class GaussianProcess:
    """GaussianProcess(; mean, kernel, lengthscale_priors, amplitude_priors, noise_std_priors)
    (gaussian_process.jl:33-41; keyword defaults from src/deprecated.jl:32-62, kernel = Matern52Kernel())."""

    def __init__(self, mean: Union[None, Sequence[float], Callable] = None, kernel=Matern52Kernel(),
                 lengthscale_priors: Optional[List[Prior]] = None, amplitude_priors: Optional[List[Prior]] = None,
                 noise_std_priors: Optional[List[Prior]] = None):
        self.mean = mean
        self.kernel = kernel
        self.lengthscale_priors = lengthscale_priors
        self.amplitude_priors = amplitude_priors
        self.noise_std_priors = noise_std_priors

    def make_discrete(self, discrete):
        base = self.kernel.kernel if isinstance(self.kernel, DiscreteKernel) else self.kernel
        k = DiscreteKernel(base, tuple(bool(b) for b in discrete)) if np.any(discrete) else base
        return GaussianProcess(self.mean, k, self.lengthscale_priors, self.amplitude_priors, self.noise_std_priors)

    # mean_getindex (gaussian_process.jl:101-103), evaluated on the host
    def mean_at(self, slice_idx: int, X):
        X = np.asarray(X, dtype=np.float64)
        if X.ndim == 1:
            X = X[:, None]
        if self.mean is None:
            return None
        if callable(self.mean):
            return np.array([np.asarray(self.mean(X[:, j]))[slice_idx] for j in range(X.shape[1])], dtype=np.float64)
        return np.full(X.shape[1], float(self.mean[slice_idx]))

    def params_sampler(self, rng):
        """_params_sampler (gaussian_process.jl:291-298)"""
        def sample():
            lam = np.stack([np.atleast_1d(p.rand(rng)) for p in self.lengthscale_priors], axis=1)
            return GaussianProcessParams(lam, np.array([p.rand(rng) for p in self.amplitude_priors]),
                                         np.array([p.rand(rng) for p in self.noise_std_priors]))
        return sample

    def params_loglike(self):
        """params_loglike (gaussian_process.jl:282-289): prior log-density, host side."""
        def ll(params: GaussianProcessParams):
            v = sum(p.logpdf(params.lengthscales[:, i]) for i, p in enumerate(self.lengthscale_priors))
            v += sum(p.logpdf(a) for p, a in zip(self.amplitude_priors, params.amplitudes))
            v += sum(p.logpdf(s) for p, s in zip(self.noise_std_priors, params.noise_std))
            return float(v)
        return ll


def _raise_domain_error(var, status):
    """The DomainError of _clip_var (gaussian_process.jl:186-194) for the first failed variance, as a ValueError."""
    if np.any(status != 0):
        bad = var[np.nonzero(status)][0]
        raise ValueError(f"DomainError: The posterior GP predicted variance {bad} but only values above -1e-8 are tolerated.")


class GaussianProcessPosterior:
    """One output slice: handle to the device-resident factor cache (replaces the AbstractGPs.PosteriorGP wrapper,
    gaussian_process.jl:127-131)."""

    def __init__(self, gp: _lib.GP, model: GaussianProcess, slice_idx: int):
        self.gp = gp
        self.model = model
        self.slice_idx = slice_idx

    def mean_and_var(self, x):
        """gaussian_process.jl:169-178: vector x -> (mu, var) scalars; matrix X -> vectors.  Raises ValueError where
        the reference throws DomainError (_clip_var)."""
        x = np.asarray(x, dtype=np.float64)
        vec = x.ndim == 1
        X = x[:, None] if vec else x
        pm = self.model.mean_at(self.slice_idx, X)
        mu, var, st = _lib.gp_predict(self.gp, X, pm)
        _raise_domain_error(var, st)
        return (float(mu[0]), float(var[0])) if vec else (mu, var)

    def mean_and_var_grad(self, x):
        """mean_and_var with the x-gradients (the mirror's stand-in for ForwardDiff through mean_and_var; one
        boss_gp_predict_grad call): vector x -> (mu, var, dmu (d,), dvar (d,)); matrix X (d x M) -> (mu (M,), var (M,),
        dmu (d, M), dvar (d, M)).  mu and var equal mean_and_var's bit for bit.  The gradient of a prior-mean closure is
        not included (the constant and zero means have none).  Raises ValueError where mean_and_var does."""
        x = np.asarray(x, dtype=np.float64)
        vec = x.ndim == 1
        X = x[:, None] if vec else x
        pm = self.model.mean_at(self.slice_idx, X)
        mu, var, dmu, dvar, st = _lib.gp_predict_grad([self.gp], 1, 1, X, None if pm is None else pm[None])
        _raise_domain_error(var, st)
        if vec:
            return float(mu[0, 0]), float(var[0, 0]), dmu[0, :, 0].copy(), dvar[0, :, 0].copy()
        return mu[0], var[0], dmu[0], dvar[0]

    def mean(self, x):
        return self.mean_and_var(x)[0]

    def var(self, x):
        return self.mean_and_var(x)[1]

    def std(self, x):
        """src/types/model_posterior.jl: std = sqrt(var)"""
        return np.sqrt(self.var(x))

    def mean_and_std(self, x):
        mu, var = self.mean_and_var(x)
        return mu, np.sqrt(var)

    def mean_and_cov(self, X):
        """gaussian_process.jl:180-184: matrix X (d x M) -> (mu (M,), Sigma (M, M)), diagonal through _clip_var."""
        X = np.asarray(X, dtype=np.float64)
        if X.ndim != 2:
            raise TypeError("cov / mean_and_cov take a matrix of points (the reference defines no vector method)")
        pm = self.model.mean_at(self.slice_idx, X)
        mu, cov, rc = _lib.gp_cov(self.gp, X, pm)
        if rc != 0:
            raise ValueError("DomainError: The posterior GP predicted a variance below -1e-8.")
        return mu, cov

    def cov(self, X):
        """gaussian_process.jl:163-167"""
        return self.mean_and_cov(X)[1]


def model_posterior_slice(model, params, data: ExperimentData, slice_idx: int) -> GaussianProcessPosterior:
    """gaussian_process.jl:133-141 / semiparametric.jl:79-84.  Raises ValueError (PosDefException) if K is not PD."""
    gp_model, gp_params = _as_gp(model, params)
    kid, mask = _kernel_parts(gp_model.kernel)
    m = gp_model.mean_at(slice_idx, data.X)
    delta = data.Y[slice_idx] - (0.0 if m is None else m)
    gp = _lib.gp_fit(data.X, delta, gp_params.lengthscales[:, slice_idx], gp_params.amplitudes[slice_idx],
                     gp_params.noise_std[slice_idx], kid, mask)
    if gp is None:
        raise ValueError("PosDefException: kernel matrix is not positive definite")
    return GaussianProcessPosterior(gp, gp_model, slice_idx)


def data_loglike(model, data: ExperimentData):
    """data_loglike(model, data) -> (params -> Real) (gaussian_process.jl:250-267, semiparametric.jl:86-92).
    The returned closure also accepts a LIST of params: one batched library call per output slice
    (the batches SamplingMAP / OptimizationMAP / TuringBI build).  Non-PD -> -inf (safe_data_loglike)."""
    def ll(params):
        single = not isinstance(params, (list, tuple))
        plist = [params] if single else list(params)
        S = len(plist)
        total = np.zeros(S)
        for i in range(data.y_dim):
            gms = [_as_gp(model, p) for p in plist]
            gp_model = gms[0][0]
            kid, mask = _kernel_parts(gp_model.kernel)
            means = [gm.mean_at(i, data.X) for gm, _ in gms]
            if all(m is None for m in means):
                Ymm = data.Y[i]
            elif not isinstance(model, Semiparametric):
                Ymm = data.Y[i] - means[0]                  # prior mean does not depend on the parameters
            else:
                Ymm = np.stack([data.Y[i] - m for m in means])
            L = np.stack([gp.lengthscales[:, i] for _, gp in gms])
            A = np.array([gp.amplitudes[i] for _, gp in gms])
            N = np.array([gp.noise_std[i] for _, gp in gms])
            total += _lib.loglik_batch(data.X, Ymm, L, A, N, kid, mask)
        return float(total[0]) if single else total
    return ll


def data_loglike_and_grad(model, data: ExperimentData):
    """(params | list of params) -> (loglik, grad): the data log-likelihood and its gradient w.r.t. the model
    parameters, shaped like the parameters: GaussianProcessParams (d lengthscales x y_dim, amplitudes, noise_std), or
    SemiparametricParams with d/dtheta in front.  What `AutoForwardDiff` gives OptimizationMAP / NUTS in the reference
    (src/model_fitters/optimization.jl:41,153), evaluated as one batched device call per output slice.
    A Semiparametric model needs Parametric(jacobian=...): its theta-gradient is alpha^T J summed over the output slices,
    J the Jacobian of the parametric mean at the training inputs (boss_gp_loglik_grad_batch_mean)."""
    semi = isinstance(model, Semiparametric)
    if semi and model.parametric.jacobian is None:
        raise NotImplementedError("data_loglike_and_grad: a Semiparametric model needs Parametric(jacobian=...)")
    gp_model = model.nonparametric if semi else model

    def llg(params):
        single = not isinstance(params, (list, tuple))
        plist = [params] if single else list(params)
        S, d, n = len(plist), data.x_dim, data.X.shape[1]
        total = np.zeros(S)
        grads = [GaussianProcessParams(np.zeros((d, data.y_dim)), np.zeros(data.y_dim), np.zeros(data.y_dim))
                 for _ in range(S)]
        kid, mask = _kernel_parts(gp_model.kernel)
        if semi:
            k = len(plist[0].theta)
            jac = model.parametric.jacobian
            # S x n x y_dim x k: d predict / d theta of every sample at every training input
            Jall = np.array([[np.asarray(jac(data.X[:, j], p.theta), dtype=np.float64).reshape(data.y_dim, k)
                              for j in range(n)] for p in plist])
            grads = [SemiparametricParams(np.zeros(k), g.lengthscales, g.amplitudes, g.noise_std) for g in grads]
        for i in range(data.y_dim):
            L = np.stack([p.lengthscales[:, i] for p in plist])
            A = np.array([p.amplitudes[i] for p in plist])
            N = np.array([p.noise_std[i] for p in plist])
            if semi:
                Ymm = np.stack([data.Y[i] - _as_gp(model, p)[0].mean_at(i, data.X) for p in plist])   # as data_loglike
                J = Jall[:, :, i, :].transpose(0, 2, 1)                                               # S x k x n
                ll, g, gm = _lib.loglik_grad_batch_mean(data.X, Ymm, J, L, A, N, kid, mask)
                for s in range(S):
                    grads[s].theta += gm[s]
            else:
                m = model.mean_at(i, data.X)
                Ymm = data.Y[i] if m is None else data.Y[i] - m
                ll, g = _lib.loglik_grad_batch(data.X, Ymm, L, A, N, kid, mask)
            total += ll
            for s in range(S):
                grads[s].lengthscales[:, i] = g[s, :d]
                grads[s].amplitudes[i] = g[s, d]
                grads[s].noise_std[i] = g[s, d + 1]
        return (float(total[0]), grads[0]) if single else (total, grads)
    return llg


# ---- Semiparametric (src/models/semiparametric.jl) ---------------------------------------------------
@dataclass
class SemiparametricParams:
    theta: np.ndarray
    lengthscales: np.ndarray
    amplitudes: np.ndarray
    noise_std: np.ndarray


class Parametric:
    """Minimal parametric model: predict(x, theta) -> y (src/models/parametric.jl); evaluated on the host.
    jacobian(x, theta), optional: the (y_dim, k) array d predict / d theta at one point -- the mirror's stand-in for the
    ForwardDiff sweep through `predict`.  With it, a Semiparametric model has data_loglike_and_grad and gradient
    OptimizationMAP."""

    def __init__(self, predict: Callable, theta_priors: Optional[List[Prior]] = None, jacobian: Optional[Callable] = None):
        self.predict = predict
        self.theta_priors = theta_priors
        self.jacobian = jacobian


class Semiparametric:
    """Semiparametric(parametric, nonparametric): the parametric prediction is the GP prior mean
    (semiparametric.jl:79-92, add_mean gaussian_process.jl:72-73)."""

    def __init__(self, parametric: Parametric, nonparametric: GaussianProcess):
        assert nonparametric.mean is None
        self.parametric = parametric
        self.nonparametric = nonparametric

    def make_discrete(self, discrete):
        return Semiparametric(self.parametric, self.nonparametric.make_discrete(discrete))

    def params_sampler(self, rng):
        gp_sample = self.nonparametric.params_sampler(rng)

        def sample():
            g = gp_sample()
            th = np.array([p.rand(rng) for p in self.parametric.theta_priors])
            return SemiparametricParams(th, g.lengthscales, g.amplitudes, g.noise_std)
        return sample

    def params_loglike(self):
        gp_ll = self.nonparametric.params_loglike()

        def ll(p: SemiparametricParams):
            v = gp_ll(GaussianProcessParams(p.lengthscales, p.amplitudes, p.noise_std))
            return v + float(sum(pr.logpdf(t) for pr, t in zip(self.parametric.theta_priors, p.theta)))
        return ll


def _as_gp(model, params):
    """Semiparametric -> GP with the parametric mean added (semiparametric.jl:79-84)."""
    if isinstance(model, Semiparametric):
        theta = params.theta
        predict = model.parametric.predict
        gpm = GaussianProcess(lambda x, _t=theta: predict(x, _t), model.nonparametric.kernel,
                              model.nonparametric.lengthscale_priors, model.nonparametric.amplitude_priors,
                              model.nonparametric.noise_std_priors)
        return gpm, GaussianProcessParams(params.lengthscales, params.amplitudes, params.noise_std)
    return model, params
