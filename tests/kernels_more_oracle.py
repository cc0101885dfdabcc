"""Reference maths for the ExponentialKernel (Matern12) and RationalQuadraticKernel GPs.

`O` is a private copy of oracle/boss_oracle.py whose covariance functions (`_kappa`, `_kappa_dr_over_r`) also accept
KERNEL_MATERN12 = 3 and an `RQ(a)` spec, so every oracle routine built on them -- posterior_fit, mean_and_var,
posterior_cov, gp_loglik(_grad), mean_var_grad, ei_acquisition, ei_value_grad, mc_ei_acquisition -- serves the new
kernels unchanged.  Distances are direct differences (see VARIANTS below).  The shared oracle module that the existing tests compare against is not modified.  Like the
oracle, this module knows nothing of the C library: RQ is described by its shape parameter, not by a registry id.

The r = 0 convention of Matern12 (DESIGN.md 2.14): kappa'(r)/r = -exp(-r)/r is taken as 0 at d2 == 0.
"""
from __future__ import annotations

import importlib.util
import os
import sys
from dataclasses import dataclass

import numpy as np

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_spec = importlib.util.spec_from_file_location("boss_oracle_kernels_more", os.path.join(_ROOT, "oracle", "boss_oracle.py"))
O = sys.modules.setdefault(_spec.name, importlib.util.module_from_spec(_spec))
if not hasattr(O, "posterior_fit"):
    _spec.loader.exec_module(O)

KERNEL_MATERN12 = 3


@dataclass(frozen=True)
class RQ:
    """RationalQuadraticKernel(alpha = a): kappa = (1 + d2 / (2a))^-a."""
    a: float


_base_kappa = O._kappa
_base_dr = O._kappa_dr_over_r


def kappa(d2, kernel):
    d2 = np.asarray(d2, dtype=np.float64)
    if isinstance(kernel, RQ):
        return np.exp(-kernel.a * np.log1p(d2 / (2.0 * kernel.a)))
    if kernel == KERNEL_MATERN12:
        return np.exp(-np.sqrt(d2))
    return _base_kappa(d2, kernel)


def kappa_dr_over_r(d2, kernel):
    d2 = np.asarray(d2, dtype=np.float64)
    if isinstance(kernel, RQ):
        return -np.exp(-(kernel.a + 1.0) * np.log1p(d2 / (2.0 * kernel.a)))
    if kernel == KERNEL_MATERN12:
        r = np.sqrt(d2)
        with np.errstate(divide="ignore", invalid="ignore"):
            return np.where(d2 == 0.0, 0.0, -np.exp(-r) / np.where(d2 == 0.0, 1.0, r))
    return _base_dr(d2, kernel)


O._kappa = kappa
O._kappa_dr_over_r = kappa_dr_over_r
# Direct coordinate differences, as the device computes them.  The GEMM form |a|^2 + |b|^2 - 2 a.b leaves a d2 of
# order 1e-16 |x|^2 for coincident points, and Matern12's sqrt turns that into an error of order 1e-8 in kappa.
O.VARIANTS["distances"] = "direct"


def _mp_kappa(mp, d2, kernel):
    if isinstance(kernel, RQ):
        a = mp.mpf(kernel.a)
        return (1 + d2 / (2 * a)) ** (-a)
    if kernel == KERNEL_MATERN12:
        return mp.e ** (-mp.sqrt(d2))
    if kernel == O.KERNEL_SE:
        return mp.e ** (-d2 / 2)
    r = mp.sqrt(d2)
    if kernel == O.KERNEL_MATERN32:
        return (1 + mp.sqrt(3) * r) * mp.e ** (-mp.sqrt(3) * r)
    if kernel == O.KERNEL_MATERN52:
        return (1 + mp.sqrt(5) * r + 5 * d2 / 3) * mp.e ** (-mp.sqrt(5) * r)
    raise ValueError(kernel)


def adjudicator_mean_var_loglik(X, y_minus_mean, lengthscales, amplitude, noise_std, kernel, Xs, dps=50):
    """oracle.adjudicator_mean_var_loglik for any of the five kernels: mu, var, loglik in `dps`-digit arithmetic with
    direct distances (n <~ 64)."""
    import mpmath as mp
    mp.mp.dps = dps
    X = np.asarray(X, dtype=np.float64); Xs = np.asarray(Xs, dtype=np.float64)
    d, n = X.shape
    M = Xs.shape[1]
    ls = [mp.mpf(float(v)) + mp.mpf('1e-8') for v in lengthscales]
    a = mp.mpf(float(amplitude)) + mp.mpf('1e-8')
    s = mp.mpf(float(noise_std)) + mp.mpf('1e-8')

    def k(p, q):
        d2 = sum(((mp.mpf(float(p[i])) - mp.mpf(float(q[i]))) / ls[i]) ** 2 for i in range(d))
        return a * a * _mp_kappa(mp, d2, kernel)

    K = mp.matrix(n, n)
    for i in range(n):
        for j in range(n):
            K[i, j] = k(X[:, i], X[:, j]) + (s * s if i == j else 0)
    L = mp.cholesky(K)
    delta = mp.matrix([mp.mpf(float(v)) for v in y_minus_mean])
    w = mp.lu_solve(L, delta)
    alpha = mp.lu_solve(L.T, w)
    logdet = 2 * sum(mp.log(L[i, i]) for i in range(n))
    ll = -(n * mp.log(2 * mp.pi) + logdet + sum(w[i] ** 2 for i in range(n))) / 2
    mu = np.empty(M); var = np.empty(M)
    for m in range(M):
        ks = mp.matrix([k(X[:, i], Xs[:, m]) for i in range(n)])
        v = mp.lu_solve(L, ks)
        mu[m] = float(sum(ks[i] * alpha[i] for i in range(n)))
        var[m] = float(a * a - sum(v[i] ** 2 for i in range(n)) + mp.mpf('1e-18'))
    return mu, var, float(ll)


def mp_kappa_and_dr(d2, kernel, dps=40):
    """kappa and kappa'(r)/r at one squared distance, from mpmath's derivative of kappa(r) (d2 > 0)."""
    import mpmath as mp
    mp.mp.dps = dps
    r0 = mp.sqrt(mp.mpf(float(d2)))
    f = lambda r: _mp_kappa(mp, r * r, kernel)
    return float(f(r0)), float(mp.diff(f, r0) / r0)


KERNELS = [KERNEL_MATERN12, RQ(0.5), RQ(2.0), RQ(50.0)]


def kernel_name(kernel) -> str:
    return f"rq{kernel.a:g}" if isinstance(kernel, RQ) else "matern12"
