"""Host twin of boss_gp_map_multistart: the numpy log-space prior (value and analytic z-gradient) and the per-slice
batched L-BFGS of acquisition_maximizers.batched_lbfgs_maximize on loglik_grad_batch + that prior."""
import math

import numpy as np

LN_SQRT_2PI = 0.5 * math.log(2.0 * math.pi)


def logprior_z(kind, par, raw):
    """kind (P,), par (P, 2), raw (S, P) raw values -> log-prior (S,) at raw and its gradient in z = log(raw) (S, P).
    Kinds: 0 Dirac (pinned: 0 and 0), 1 Normal(mu, s), 2 LogNormal(mu, s), 3 Uniform(lo, hi) inclusive."""
    raw = np.atleast_2d(np.asarray(raw, dtype=np.float64))
    S, P = raw.shape
    lp = np.zeros(S)
    dz = np.zeros((S, P))
    with np.errstate(divide="ignore", invalid="ignore"):
        for j in range(P):
            a, b = par[j]
            x = raw[:, j]
            if kind[j] == 1:
                r = (x - a) / b
                lp += -0.5 * r * r - (math.log(b) + LN_SQRT_2PI)
                dz[:, j] = -r / b * x
            elif kind[j] == 2:
                r = (np.log(x) - a) / b
                lp += -0.5 * r * r - np.log(x * b * math.sqrt(2 * math.pi))
                dz[:, j] = -r / b - 1.0
            elif kind[j] == 3:
                lp += np.where((a <= x) & (x <= b), -math.log(b - a), -np.inf)
    return lp, dz


def raw_of(kind, par, Z):
    """z (S, P) -> raw (S, P): exp(z), or the pinned value of a Dirac entry."""
    return np.where(np.asarray(kind)[None, :] == 0, np.asarray(par)[None, :, 0], np.exp(Z))


def z_of(kind, starts):
    """raw starts (S, P) -> z (S, P): log for the free entries, 0 for the pinned ones."""
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.where(np.asarray(kind)[None, :] == 0, 0.0, np.log(starts))


def value_and_grad(lib, X, y, kind, par, kernel_id, mask=None):
    """One slice's objective as batched_lbfgs_maximize takes it: Z (P, m) -> f (m,), G (P, m)."""
    d = X.shape[0]

    def vg(Z):
        raw = raw_of(kind, par, np.asarray(Z).T)
        ll, g = lib.loglik_grad_batch(X, y, raw[:, :d], raw[:, d], raw[:, d + 1], kernel_id, mask)
        lp, dz = logprior_z(kind, par, raw)
        f = ll + lp
        G = np.where(np.asarray(kind)[None, :] == 0, 0.0, raw * g + dz)
        bad = ~np.isfinite(f)
        f[bad] = -np.inf
        G[bad] = 0.0
        return f, G.T
    return vg


def host_twin(lib, X, Ymm, kind, par, starts, kernel_id, mask=None, iters=40, history=8):
    """Per slice: batched_lbfgs_maximize in z inside [-30, 30].  -> raw params (y_dim, M, P), f (y_dim, M)."""
    from boss_b200.acquisition_maximizers import batched_lbfgs_maximize
    y_dim, M, P = starts.shape
    po = np.empty_like(starts)
    fo = np.empty((y_dim, M))
    lo, hi = np.full(P, -30.0), np.full(P, 30.0)
    for i in range(y_dim):
        vg = value_and_grad(lib, X, Ymm[i], kind[i], par[i], kernel_id, mask)
        Z, f = batched_lbfgs_maximize(vg, z_of(kind[i], starts[i]).T, lo, hi, iters=iters, history=history)
        po[i] = raw_of(kind[i], par[i], Z.T)
        fo[i] = f
    return po, fo


def start_values(lib, X, Ymm, kind, par, starts, kernel_id, mask=None):
    """The objective at the (clipped) starts, (y_dim, M)."""
    out = np.empty(starts.shape[:2])
    for i in range(starts.shape[0]):
        vg = value_and_grad(lib, X, Ymm[i], kind[i], par[i], kernel_id, mask)
        out[i] = vg(np.clip(z_of(kind[i], starts[i]), -30.0, 30.0).T)[0]
    return out
