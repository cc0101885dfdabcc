"""Host-side mirror of the BOSS.jl types that sit on the accelerated path (names and argument meaning
follow the reference: src/types/*.jl).  Pure Python / numpy: no numerics of the hot path live here."""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import Callable, List, Optional, Sequence

import numpy as np


# ---- Domain (src/types/domain.jl:30-84) -----------------------------------------------------------
class Domain:
    def __init__(self, bounds, discrete=None, cons: Optional[Callable] = None):
        lb, ub = bounds
        self.bounds = (np.asarray(lb, dtype=np.float64), np.asarray(ub, dtype=np.float64))
        d = self.bounds[0].shape[0]
        self.discrete = np.zeros(d, dtype=bool) if discrete is None else np.asarray(discrete, dtype=bool)
        assert self.bounds[0].shape == self.bounds[1].shape == self.discrete.shape      # domain.jl:41
        if cons is not None and self.discrete.any():                                       # make_discrete, :52-61
            raw, disc = cons, self.discrete
            cons = lambda x: raw(discrete_round(disc, x))
        self.cons = cons

    @property
    def x_dim(self):
        return self.discrete.shape[0]


def discrete_round(dims, x):
    """src/utils/utils.jl:24-26 (Julia `round` = ties-to-even = numpy.rint)."""
    x = np.array(x, dtype=np.float64, copy=True)
    if dims is None:
        return x
    dims = np.asarray(dims, dtype=bool)
    x[dims] = np.rint(x[dims])
    return x


def in_bounds(x, bounds):
    """domain.jl:73-78 (inclusive).  x: (d,) or (d, M) -> bool or (M,)"""
    x = np.asarray(x, dtype=np.float64)
    lb, ub = bounds
    if x.ndim == 1:
        return not (np.any(x < lb) or np.any(x > ub))
    return ~(np.any(x < lb[:, None], axis=0) | np.any(x > ub[:, None], axis=0))


def in_discrete(x, discrete):
    x = np.asarray(x, dtype=np.float64)
    return bool(np.all(np.rint(x[discrete]) == x[discrete]))


def in_cons(x, cons):
    """domain.jl:83-84: all(cons(x) .>= 0)"""
    return True if cons is None else bool(np.all(np.asarray(cons(x)) >= 0.0))


def in_domain(x, domain: Domain):
    return in_bounds(x, domain.bounds) and in_discrete(x, domain.discrete) and in_cons(x, domain.cons)


def cons_mask(X, domain: Domain):
    """Evaluate the user's `cons` closure on the host for every column (the C ABI takes the byte mask)."""
    if domain.cons is None:
        return None
    X = np.asarray(X, dtype=np.float64)
    return np.fromiter((in_cons(X[:, j], domain.cons) for j in range(X.shape[1])), dtype=np.uint8, count=X.shape[1])


# ---- Fitness (src/types/fitness.jl) ---------------------------------------------------------------
@dataclass
class LinFitness:
    coefs: Sequence[float]

    def __call__(self, y):
        return float(np.asarray(self.coefs, dtype=np.float64) @ np.asarray(y, dtype=np.float64))


@dataclass
class NonlinFitness:
    """fitness(y) -> Real.  `grad` (optional): grad(Y) -> df/dy (y_dim x P) at the columns of a y_dim x P matrix Y --
    what ForwardDiff does to the closure in the reference.  With it, Acquisition.value_and_grad (and so OptimizationAM
    and SampleOptAM) can differentiate the Monte-Carlo EI of the closure; the closure itself stays on the host."""
    fitness: Callable
    grad: Optional[Callable] = None

    def __call__(self, y):
        return self.fitness(y)


class ExprFitness(NonlinFitness):
    """A NonlinFitness from the small expression set the device can evaluate (include/boss_b200.h, boss_mcei_score):
         kind "affine"     f(y) = c0 + c . y
              "quadratic"  f(y) = c0 + c . y + sum_i q_i (y_i - t_i)^2
              "max"/"min"  f(y) = c0 + max/min over {i : c_i != 0} of (c_i y_i + t_i)
    It is an ordinary fitness closure on the host (so best_so_far etc. work unchanged); ExpectedImprovement with it runs
    the Monte-Carlo EI of expected_improvement.jl:104-111 on the device instead of finishing it on the host."""
    KINDS = {"affine": 1, "quadratic": 2, "max": 3, "min": 4}

    def __init__(self, kind: str, c, c0: float = 0.0, q=None, t=None):
        self.kind = kind
        self.kind_id = self.KINDS[kind]
        self.c = np.asarray(c, dtype=np.float64)
        self.c0 = float(c0)
        self.q = np.zeros_like(self.c) if q is None else np.asarray(q, dtype=np.float64)
        self.t = np.zeros_like(self.c) if t is None else np.asarray(t, dtype=np.float64)
        super().__init__(self._eval)

    def _eval(self, y):
        y = np.asarray(y, dtype=np.float64)
        cy = self.c[:, None] * y if y.ndim == 2 else self.c * y
        if self.kind_id == 1:
            return self.c0 + cy.sum(axis=0)
        if self.kind_id == 2:
            dv = y - (self.t[:, None] if y.ndim == 2 else self.t)
            return self.c0 + cy.sum(axis=0) + ((self.q[:, None] if y.ndim == 2 else self.q) * dv * dv).sum(axis=0)
        live = self.c != 0
        v = (cy + (self.t[:, None] if y.ndim == 2 else self.t))[live]
        return self.c0 + (v.max(axis=0) if self.kind_id == 3 else v.min(axis=0))


# ---- data (src/data/simple_data.jl) ---------------------------------------------------------------
class ExperimentData:
    def __init__(self, X, Y):
        self.X = np.asarray(X, dtype=np.float64).reshape(np.shape(X)[0], -1)     # x_dim x n
        self.Y = np.asarray(Y, dtype=np.float64).reshape(np.shape(Y)[0], -1)     # y_dim x n
        assert self.X.shape[1] == self.Y.shape[1]

    def augment(self, X, Y):
        """augment_dataset! (src/data/simple_data.jl:24-29): hcat new columns."""
        X = np.asarray(X, dtype=np.float64).reshape(self.X.shape[0], -1)
        Y = np.asarray(Y, dtype=np.float64).reshape(self.Y.shape[0], -1)
        self.X = np.concatenate([self.X, X], axis=1)
        self.Y = np.concatenate([self.Y, Y], axis=1)

    @property
    def x_dim(self):
        return self.X.shape[0]

    @property
    def y_dim(self):
        return self.Y.shape[0]

    def __len__(self):
        return self.X.shape[1]


# ---- fitted parameters (src/types/parameters.jl) ----------------------------------------------------
@dataclass
class MAPParams:
    params: object
    loglike: float


@dataclass
class BIParams:
    samples: list            # Vector{ModelParams}


@dataclass
class FixedParams:
    params: object


def get_params(p):
    if isinstance(p, BIParams):
        return p.samples
    if isinstance(p, (MAPParams, FixedParams)):
        return p.params
    return p


@dataclass
class BossOptions:
    info: bool = False
    debug: bool = False
    callback: Optional[Callable] = None


class BossProblem:
    """src/types/problem.jl:38-80"""

    def __init__(self, f, domain: Domain, acquisition, model, data: ExperimentData, y_max=None, params=None):
        assert domain.x_dim == data.x_dim                                         # problem.jl:51
        self.f = f
        self.domain = domain
        self.y_max = np.full(data.y_dim, np.inf) if y_max is None else np.asarray(y_max, dtype=np.float64)
        assert self.y_max.shape[0] == data.y_dim
        self.acquisition = acquisition
        self.model = model.make_discrete(domain.discrete) if domain.discrete.any() else model
        self.params = FixedParams(params) if (params is not None and not isinstance(params, (MAPParams, BIParams, FixedParams))) else params
        self.data = data
        self.consistent = False


# ---- priors (host-side prior plumbing: O(#params), out of the hot path) ---------------------------------
class Prior:
    def rand(self, rng):
        raise NotImplementedError

    def logpdf(self, x):
        raise NotImplementedError


@dataclass
class LogNormal(Prior):
    mu: float = 0.0
    sigma: float = 1.0

    def rand(self, rng):
        return float(np.exp(rng.normal(self.mu, self.sigma)))

    def logpdf(self, x):
        if x <= 0:
            return -math.inf
        z = (math.log(x) - self.mu) / self.sigma
        return -0.5 * z * z - math.log(x * self.sigma * math.sqrt(2 * math.pi))


@dataclass
class Normal(Prior):
    mu: float = 0.0
    sigma: float = 1.0

    def rand(self, rng):
        return float(rng.normal(self.mu, self.sigma))

    def logpdf(self, x):
        z = (x - self.mu) / self.sigma
        return -0.5 * z * z - math.log(self.sigma * math.sqrt(2 * math.pi))


@dataclass
class Uniform(Prior):
    lo: float
    hi: float

    def rand(self, rng):
        return float(rng.uniform(self.lo, self.hi))

    def logpdf(self, x):
        return -math.log(self.hi - self.lo) if self.lo <= x <= self.hi else -math.inf


@dataclass
class Dirac(Prior):
    value: float

    def rand(self, rng):
        return float(self.value)

    def logpdf(self, x):
        return 0.0 if x == self.value else -math.inf


@dataclass
class Product(Prior):
    """Multivariate prior with independent components (e.g. BOSS.mvlognormal)."""
    parts: List[Prior]

    def rand(self, rng):
        return np.array([p.rand(rng) for p in self.parts])

    def logpdf(self, x):
        return float(sum(p.logpdf(v) for p, v in zip(self.parts, x)))


def mvlognormal(mu, sigma):
    return Product([LogNormal(float(m), float(s)) for m, s in zip(mu, sigma)])


def generate_LHC(bounds, count, rng):
    """Latin hypercube starts (src/utils/utils.jl:52-58): one stratum per point per dimension."""
    lb, ub = bounds
    d = lb.shape[0]
    out = np.empty((d, count))
    for i in range(d):
        perm = rng.permutation(count)
        out[i] = lb[i] + (perm + rng.random(count)) / count * (ub[i] - lb[i])
    return out
