"""References for the batched log-likelihood family at the sizes it runs at (n up to a few thousand, S up to tens of
thousands), and a mirror of how `loglik_core` (boss.jl_b200/csrc/boss_b200.cu) cuts a batch into workspace windows and
stream groups.

- `adjudicator_grad_longdouble`: log-likelihood and its hyper-parameter gradient in x87 extended precision (numpy
  longdouble, 64-bit mantissa): direct distances, the column Cholesky written out, alpha, K^-1 = W^T W with W = L^-1,
  and 1/2 sum((alpha alpha^T - K^-1) o dK/dtheta) ordered [lengthscales; amplitude; noise_std].  It extends
  oracle.adjudicator_longdouble to the gradient and to all five covariance functions (tests/kernels_more_oracle.py's
  kappa, with Matern-1/2's kappa'(r)/r = 0 at r = 0), discrete dimensions included.
- `reference_grad`: the FP64 reference the GPU tests compare with (oracle.gp_loglik_grad, through kernels_more_oracle's
  copy for Matern-1/2 and RQ), and `grad_ratio`, the comparison those tests apply.
- `window_plan`: the sample windows and stream groups loglik_core runs a batch as.
"""
from __future__ import annotations

import math

import numpy as np

from oracle import boss_oracle as OB
from tests.kernels_more_oracle import KERNEL_MATERN12, RQ, O as OK

TM = 128                                     # csrc/common.cuh `TM`, rows of a block
LL_GROUPS = 16                               # csrc/boss_b200.cu `LL_GROUPS`, most stream groups a window runs as
WORKSPACE_BYTES = 32 << 30                   # loglik_core's workspace budget for a window (`Sb`)
MAX_WINDOW = 32768                           # loglik_core's cap on `Sb`
SMALL_N = 32                                 # csrc/tk_params.cuh `SMALL_N`, warp-register path (value mode only)
TOL_LL, TOL_GRAD, TOL_JAC, TOL_POST = 1e-8, 1e-8, 1e-9, 1e-9


# ---- references ----------------------------------------------------------------------------------------------------

def oracle_for(kernel):
    """The shared oracle for SE / Matern-3/2 / Matern-5/2, kernels_more_oracle's extended copy for the others."""
    return OB if kernel in (OB.KERNEL_SE, OB.KERNEL_MATERN32, OB.KERNEL_MATERN52) else OK


def reference_grad(X, y_minus_mean, ls, amp, noise, kernel, mask=None):
    return oracle_for(kernel).gp_loglik_grad(X, y_minus_mean, ls, amp, noise, kernel, mask)


def grad_ratio(g, ref, tol=TOL_GRAD):
    """max_i |g_i - ref_i| / (tol * |ref|_2): the GPU tests' gradient check passes when this is <= 1."""
    g, ref = np.asarray(g, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    return float(np.max(np.abs(g - ref))) / (tol * max(float(np.linalg.norm(ref)), 1e-300))


def rel_ratio(v, ref, tol=TOL_LL):
    return abs(float(v) - float(ref)) / (tol * max(abs(float(ref)), 1e-300))


def _kappa_ld(D2, kernel):
    """kappa and kappa'(r)/r in long double."""
    LD = np.longdouble
    if isinstance(kernel, RQ):
        a = LD(kernel.a)
        lp = np.log1p(D2 / (2 * a))
        return np.exp(-a * lp), -np.exp(-(a + 1) * lp)
    if kernel == OB.KERNEL_SE:
        e = np.exp(-D2 / LD(2))
        return e, -e
    r = np.sqrt(D2)
    if kernel == OB.KERNEL_MATERN32:
        c = np.sqrt(LD(3))
        e = np.exp(-c * r)
        return (1 + c * r) * e, -3 * e
    if kernel == OB.KERNEL_MATERN52:
        c = np.sqrt(LD(5))
        e = np.exp(-c * r)
        return (1 + c * r + LD(5) * D2 / LD(3)) * e, -(LD(5) / LD(3)) * (1 + c * r) * e
    if kernel == KERNEL_MATERN12:
        e = np.exp(-r)
        zero = D2 == 0
        return e, np.where(zero, LD(0), -e / np.where(zero, LD(1), r))
    raise ValueError(kernel)


def adjudicator_grad_longdouble(X, y_minus_mean, lengthscales, amplitude, noise_std, kernel, discrete_mask=None):
    """-> (loglik, grad (d + 2,)) as float64 roundings of the extended-precision values; (-inf, zeros) when the column
    Cholesky meets a non-positive pivot.  Cost ~ 7/6 n^3 long-double multiply-adds (n = 1000: a few seconds)."""
    LD = np.longdouble
    X = OB.discrete_round(discrete_mask, np.asarray(X, dtype=np.float64)).astype(LD)
    d, n = X.shape
    ls = np.asarray(lengthscales, dtype=np.float64).astype(LD) + LD(OB.MIN_PARAM_VALUE)
    a = LD(float(amplitude)) + LD(OB.MIN_PARAM_VALUE)
    s = LD(float(noise_std)) + LD(OB.MIN_PARAM_VALUE)
    Xa = X / ls[:, None]
    D2 = np.zeros((n, n), dtype=LD)
    for q in range(d):
        diff = Xa[q][:, None] - Xa[q][None, :]
        D2 += diff * diff
    Kc, g = _kappa_ld(D2, kernel)
    K = a * a * Kc
    K[np.diag_indices(n)] += s * s
    L = np.zeros((n, n), dtype=LD)
    for j in range(n):                                   # column Cholesky
        v = K[j:, j] - L[j:, :j] @ L[j, :j]
        if not v[0] > 0:
            return -math.inf, np.zeros(d + 2)
        L[j, j] = np.sqrt(v[0])
        L[j + 1:, j] = v[1:] / L[j, j]
    W = np.zeros((n, n), dtype=LD)                       # W = L^-1 (lower), row by row
    for i in range(n):
        W[i, i] = 1 / L[i, i]
        if i:
            W[i, :i] = -(L[i, :i] @ W[:i, :i]) / L[i, i]
    delta = np.asarray(y_minus_mean, dtype=np.float64).astype(LD)
    w = W @ delta
    alpha = W.T @ w
    ll = -(n * np.log(2 * np.pi * LD(1)) + 2 * np.sum(np.log(np.diag(L))) + np.sum(w * w)) / 2
    G = np.outer(alpha, alpha) - W.T @ W                 # alpha alpha^T - K^-1
    grad = np.empty(d + 2, dtype=LD)
    Gg = G * g
    for q in range(d):
        dq2 = (Xa[q][:, None] - Xa[q][None, :]) ** 2
        grad[q] = -a * a * np.sum(Gg * dq2) / (2 * ls[q])
    grad[d] = a * np.sum(G * Kc)
    grad[d + 1] = np.trace(G) * s
    return float(ll), grad.astype(np.float64)


def mp_loglik_grad(X, y_minus_mean, lengthscales, amplitude, noise_std, kernel, discrete_mask=None, dps=40):
    """40-digit reference (n <~ 12): the log-likelihood in mpmath, differentiated by mp.diff in each raw
    hyper-parameter."""
    import mpmath as mp
    from tests.kernels_more_oracle import _mp_kappa
    mp.mp.dps = dps
    X = OB.discrete_round(discrete_mask, np.asarray(X, dtype=np.float64))
    d, n = X.shape
    Xm = [[mp.mpf(float(X[q, i])) for i in range(n)] for q in range(d)]
    dm = [mp.mpf(float(v)) for v in y_minus_mean]
    eps = mp.mpf(OB.MIN_PARAM_VALUE)

    def ll(theta):
        ls = [theta[q] + eps for q in range(d)]
        a, s = theta[d] + eps, theta[d + 1] + eps
        K = mp.matrix(n, n)
        for i in range(n):
            for j in range(n):
                d2 = sum(((Xm[q][i] - Xm[q][j]) / ls[q]) ** 2 for q in range(d))
                K[i, j] = a * a * _mp_kappa(mp, d2, kernel) + (s * s if i == j else 0)
        L = mp.cholesky(K)
        w = mp.lu_solve(L, mp.matrix(dm))
        return -(n * mp.log(2 * mp.pi) + 2 * sum(mp.log(L[i, i]) for i in range(n)) + sum(w[i] ** 2 for i in range(n))) / 2

    theta0 = [mp.mpf(float(v)) for v in lengthscales] + [mp.mpf(float(amplitude)), mp.mpf(float(noise_std))]
    grad = np.empty(d + 2)
    for c in range(d + 2):
        def f(t, c=c):
            th = list(theta0)
            th[c] = t
            return ll(th)
        grad[c] = float(mp.diff(f, theta0[c]))
    return float(ll(theta0)), grad


def tile_contributions(X, y_minus_mean, lengthscales, amplitude, noise_std, kernel, discrete_mask=None):
    """The FP64 reference gradient split by 128 x 128 tile of G = alpha alpha^T - K^-1 (the tiles loglik_grad_tile_kernel
    sums): -> (grad (d + 2,), part (nblk, nblk, d + 2)) with grad == part.sum((0, 1)) up to rounding.  Dropping part[i, j]
    from the sum is the gradient of a kernel that skipped that tile."""
    import scipy.linalg as sl
    Om = oracle_for(kernel)
    X = np.asarray(X, dtype=np.float64)
    ls, amp, noise = OB.condition_params(lengthscales, amplitude, noise_std)
    d, n = X.shape
    Xa = OB.discrete_round(discrete_mask, X) / ls[:, None]
    D2 = OB._pairwise_sqdist_direct(Xa, Xa)
    Kc = Om._kappa(D2, kernel)
    K = amp * amp * Kc
    K[np.diag_indices(n)] += noise * noise
    U = OB.cholesky_upper(K)
    alpha = sl.cho_solve((U, False), np.asarray(y_minus_mean, dtype=np.float64), check_finite=False)
    G = np.outer(alpha, alpha) - sl.cho_solve((U, False), np.eye(n), check_finite=False)
    Gg = G * Om._kappa_dr_over_r(D2, kernel)
    nblk = (n + TM - 1) // TM
    part = np.zeros((nblk, nblk, d + 2))
    grad = np.empty(d + 2)
    for c in range(d + 2):
        if c < d:
            T = 0.5 * Gg * (-amp * amp * (Xa[c][:, None] - Xa[c][None, :]) ** 2 / ls[c])
        elif c == d:
            T = 0.5 * G * (2.0 * amp * Kc)
        else:
            T = np.diag(np.diag(G)) * noise
        grad[c] = T.sum()
        for bi in range(nblk):
            for bj in range(nblk):
                part[bi, bj, c] = T[bi * TM:(bi + 1) * TM, bj * TM:(bj + 1) * TM].sum()
    return grad, part


# ---- windows and stream groups -------------------------------------------------------------------------------------

def window_plan(n, d, S, mode, groups=None, timing=False):
    """The windows and stream groups loglik_core runs a batch of S samples as (a name in a comment: the loglik_core
    variable the line mirrors).

    mode: "value" (boss_gp_loglik_batch), "grad" (the gradient entry points) or "fit" (boss_gp_fit_batch).
    groups: BOSS_LL_GROUPS, None when unset.  timing: boss_set_timing(1).
    -> dict(Sb=..., small=..., windows=[dict(s0, sb, ngroups, gsz, groups=[(so, gs), ...]), ...])."""
    n_pad = (n + TM - 1) // TM * TM
    nblk = n_pad // TM
    mat = n_pad * n_pad
    need_w = mode in ("grad", "fit")                                       # need_w
    small = n <= SMALL_N and not need_w                                    # small
    per = (3 if need_w else 1) * mat * 8 + (2 * nblk if need_w else nblk) * TM * TM * 8   # per
    Sb = max(1, min(S, WORKSPACE_BYTES // per))                            # Sb
    Sb = min(Sb, MAX_WINDOW)
    if small:                                                              # one launch for the whole batch
        return dict(Sb=1, small=True, per=per, windows=[])
    windows = []
    for s0 in range(0, S, Sb):                                             # the window loop
        sb = min(Sb, S - s0)
        want = 2 if nblk <= 6 else 4                                       # want_groups
        if groups is not None:
            want = max(1, min(LL_GROUPS, int(groups)))
        ngroups = 1 if (timing or sb < 2 * want) else want                 # ngroups
        gsz = (sb + ngroups - 1) // ngroups                                # gsz
        gl = []
        for gi in range(ngroups):                                          # the group loop: wo, gs
            wo = gi * gsz
            gs = min(gsz, sb - wo)
            if gs <= 0:
                break
            gl.append((s0 + wo, gs))
        windows.append(dict(s0=s0, sb=sb, ngroups=ngroups, gsz=gsz, groups=gl))
    return dict(Sb=Sb, small=False, per=per, windows=windows)


def boundary_samples(plan):
    """The first and last sample of every group of every window."""
    out = set()
    for w in plan["windows"]:
        for so, gs in w["groups"]:
            out.update((so, so + gs - 1))
    return sorted(out)
