"""numpy reference of the prior-mean gradient of the log marginal likelihood (DESIGN.md 2.13, include/boss_b200.h
boss_gp_loglik_grad_batch_mean), built on the oracle's kernel matrix and Cholesky factor:

    d LML / d theta_c = alpha^T J[:, c],   alpha = K^-1 (y - m(X; theta)),   J = dm(X; theta)/dtheta

with alpha from the same two triangular solves O.gp_loglik_grad forms it with.  The CPU tests check it against central
differences of O.gp_loglik, the GPU tests check the device against it."""
import math

import numpy as np
import scipy.linalg as sl

from oracle import boss_oracle as O


def gp_loglik_mean_grad(X, y_minus_mean, J, lengthscales, amplitude, noise_std, kernel_id=O.KERNEL_MATERN52,
                        discrete_mask=None):
    """J (k, n) -> (ll, alpha^T J (k,)); (-inf, zeros) when K is not positive definite."""
    X = np.asarray(X, dtype=np.float64)
    delta = np.asarray(y_minus_mean, dtype=np.float64)
    J = np.asarray(J, dtype=np.float64)
    ls, amp, noise = O.condition_params(lengthscales, amplitude, noise_std)
    n = X.shape[1]
    K = O.kernel_matrix(X, None, ls, amp, kernel_id, discrete_mask)
    K[np.diag_indices(n)] += noise * noise
    try:
        U = O.cholesky_upper(K)
    except O.PosDefException:
        return -math.inf, np.zeros(J.shape[0])
    w = sl.solve_triangular(U, delta, trans='T', lower=False, check_finite=False)
    alpha = sl.solve_triangular(U, w, trans='N', lower=False, check_finite=False)
    ll = float(-(n * O.LOG2PI + 2.0 * np.sum(np.log(np.diag(U))) + np.dot(w, w)) / 2.0)
    return ll, J @ alpha


def gp_loglik_mean_grad_batch(X, Y_minus_mean, J, lengthscales, amplitude, noise_std, kernel_id=O.KERNEL_MATERN52,
                              discrete_mask=None):
    """Y_minus_mean (n,) or (S, n); J (k, n) shared or (S, k, n) -> ll (S,), grad_mean (S, k)."""
    lengthscales = np.asarray(lengthscales, dtype=np.float64)
    S = lengthscales.shape[0]
    Ym = np.asarray(Y_minus_mean, dtype=np.float64)
    J = np.asarray(J, dtype=np.float64)
    ll = np.empty(S); gm = np.empty((S, J.shape[-2]))
    for s in range(S):
        ll[s], gm[s] = gp_loglik_mean_grad(X, Ym if Ym.ndim == 1 else Ym[s], J if J.ndim == 2 else J[s], lengthscales[s],
                                           amplitude[s], noise_std[s], kernel_id, discrete_mask)
    return ll, gm
