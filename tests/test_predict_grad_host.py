"""The host chain rule of a NonlinFitness closure with `grad` (boss_b200.acquisition.mc_ei_value_grad, DESIGN.md 2.12),
without a GPU: fed the oracle's mean_var_grad outputs, it must give the numpy reference of the device's Monte-Carlo EI
gradient (tests/mcei_grad_oracle.py) for the four expression kinds, and central differences of the oracle's
Monte-Carlo EI for a closure outside the expression set."""
import numpy as np
import pytest

from oracle import boss_oracle as O
from tests import mcei_grad_oracle as MO
from tests.util_problems import make_problem


def _helper():
    from boss_b200.acquisition import mc_ei_value_grad
    return mc_ei_value_grad


EXPR = {1: (1.0, [0.7, -0.2], [0.0, 0.0], [0.0, 0.0]),
        2: (0.1, [1.0, 0.3], [0.0, -0.5], [0.0, 0.2]),
        3: (0.0, [1.0, 0.8], [0.0, 0.0], [0.0, 0.1]),
        4: (0.0, [1.0, 2.0], [0.0, 0.0], [0.0, 0.5])}


def _posts(S, y_dim=2, n=30, d=3, seed=0):
    X, Y, ls, amp, ns = make_problem(n, d, seed=seed, y_dim=y_dim)
    posts = [[O.posterior_fit(X, Y[i], ls[i] * (1 + 0.15 * s), amp[i], ns[i], O.KERNEL_MATERN52) for i in range(y_dim)]
             for s in range(S)]
    return X, Y, posts


def _stack(posts, Xs, pm=None, pmg=None):
    """The oracle's mean_var_grad of every posterior, shaped as the helper takes them: (S, y_dim, ...)."""
    S, y_dim = len(posts), len(posts[0])
    out = [[O.mean_var_grad(posts[s][i], Xs, None if pm is None else pm[i], None if pmg is None else pmg[i])
            for i in range(y_dim)] for s in range(S)]
    return tuple(np.array([[out[s][i][k] for i in range(y_dim)] for s in range(S)]) for k in range(5))


def _grad_err(grad, gref):
    scale = np.max(np.abs(gref), axis=1, keepdims=True)
    scale = np.where(scale > 0, scale, 1.0)
    return float(np.max(np.abs(grad - gref) / scale))


@pytest.mark.parametrize("kind", [1, 2, 3, 4])
@pytest.mark.parametrize("with_ymax", [False, True])
@pytest.mark.parametrize("S", [1, 3])
def test_helper_matches_the_expression_reference(kind, with_ymax, S):
    """The chain rule with f, g of an expression kind equals the numpy reference of the device's MC-EI gradient; a
    linear prior mean on output 0 with its gradient."""
    mc_ei_value_grad = _helper()
    d, M = 3, 40
    X, Y, posts = _posts(S, seed=40 + kind)
    rng = np.random.default_rng(kind + 10 * S)
    eps = rng.standard_normal((2, 64 if S == 1 else S))
    c0, c, q, t = (np.asarray(v, dtype=np.float64) if isinstance(v, list) else v for v in EXPR[kind])
    fY = lambda Z: MO._fit_and_grad(kind, c0, c, q, t, Z)[0]
    gY = lambda Z: MO._fit_and_grad(kind, c0, c, q, t, Z)[1]
    f1 = MO.fitness(kind, c0, c, q, t)
    best = float(np.quantile([f1(Y[:, j]) for j in range(Y.shape[1])], 0.5))
    y_max = np.array([np.inf, float(np.quantile(Y[1], 0.6))]) if with_ymax else None
    Xs = rng.random((d, M))
    theta = np.array([0.3, -0.2, 0.1])
    pm = np.stack([theta @ Xs, np.zeros(M)])
    pmg = np.zeros((2, d, M))
    pmg[0] = theta[:, None]
    mu, var, dmu, dvar, st = _stack(posts, Xs, pm, pmg)
    val, grad = mc_ei_value_grad(mu, var, dmu, dvar, eps, fY, gY, best, y_max, status=st)
    vref, gref = MO.mc_ei_value_grad(posts, Xs, kind, c0, c, q, t, eps, best, y_max, pm, pmg)
    assert np.any(vref > 0) and np.any(gref != 0)
    assert np.allclose(val, vref, rtol=1e-12, atol=1e-300)
    assert _grad_err(grad, gref) <= 1e-12


def _cos_sin():
    f = lambda Z: np.cos(Z[0]) + np.sin(Z[1])                          # the reference's NonlinFitness docstring example
    g = lambda Z: np.stack([-np.sin(Z[0]), np.cos(Z[1])])
    return f, g


@pytest.mark.parametrize("with_ymax", [False, True])
@pytest.mark.parametrize("S", [1, 3])
def test_helper_matches_central_differences_for_a_closure(with_ymax, S):
    """f(y) = cos(y0) + sin(y1) is outside the expression set: the helper's value equals the oracle's Monte-Carlo EI,
    and its gradient central differences of it.  Candidates within 1e-4 of a kink (some |imp_k|) are skipped."""
    mc_ei_value_grad = _helper()
    d, M = 3, 24
    X, Y, posts = _posts(S, seed=7)
    f, g = _cos_sin()
    best = float(np.quantile(f(Y), 0.5))
    rng = np.random.default_rng(11 + S)
    eps = rng.standard_normal((2, 64 if S == 1 else S))
    y_max = np.array([np.inf, float(np.quantile(Y[1], 0.6))]) if with_ymax else None
    Xs = rng.random((d, M))
    mu, var, dmu, dvar, st = _stack(posts, Xs)
    val, grad = mc_ei_value_grad(mu, var, dmu, dvar, eps, f, g, best, y_max, status=st)
    f1 = lambda y: float(np.cos(y[0]) + np.sin(y[1]))
    ref = O.mc_ei_acquisition(posts, Xs, f1, eps, best, y_max)
    assert np.any(ref > 0)
    assert np.allclose(val, ref, rtol=1e-10, atol=1e-300)   # PoF deep in the tail: erfc implementations differ
    margin = np.full(M, np.inf)                     # distance of every candidate's improvements from 0
    for s in range(S):
        e = eps if S == 1 else eps[:, s:s + 1]
        Yk = mu[s][:, :, None] + np.sqrt(var[s])[:, :, None] * e[:, None, :]
        margin = np.minimum(margin, np.min(np.abs(f(Yk) - best), axis=1))
    keep = margin > 1e-4
    assert keep.sum() >= M // 2 and np.any(grad[:, keep] != 0.0)
    h = 1e-6
    for j in range(d):
        Xp = Xs.copy(); Xp[j] += h
        Xm = Xs.copy(); Xm[j] -= h
        fd = (O.mc_ei_acquisition(posts, Xp, f1, eps, best, y_max) - O.mc_ei_acquisition(posts, Xm, f1, eps, best, y_max)) / (2 * h)
        assert np.allclose(grad[j, keep], fd[keep], rtol=2e-5, atol=1e-9), (j, grad[j, keep], fd[keep])


def test_helper_conventions_nan_failed_and_pof_only():
    """A NaN improvement gives a NaN gradient; a failed variance gives -inf and a zero gradient; best = None gives PoF
    and its gradient alone (the oracle's closed form with best = None)."""
    mc_ei_value_grad = _helper()
    d, M = 3, 12
    X, Y, posts = _posts(1, seed=3)
    f, g = _cos_sin()
    eps = np.random.default_rng(2).standard_normal((2, 16))
    Xs = np.random.default_rng(4).random((d, M))
    mu, var, dmu, dvar, st = _stack(posts, Xs)
    fn = lambda Z: np.where(np.arange(Z.shape[1]) // 16 == 2, np.nan, f(Z))   # candidate 2: NaN fitness
    val, grad = mc_ei_value_grad(mu, var, dmu, dvar, eps, fn, g, -10.0, None, status=st)
    assert np.isnan(val[2]) and np.all(np.isnan(grad[:, 2]))
    assert np.all(np.isfinite(val[[0, 1, 3]])) and np.all(np.isfinite(grad[:, [0, 1, 3]]))
    st2 = st.copy()
    st2[0, 1, 5] = 2
    val, grad = mc_ei_value_grad(mu, var, dmu, dvar, eps, f, g, -10.0, None, status=st2)
    assert np.isneginf(val[5]) and np.all(grad[:, 5] == 0.0) and np.all(np.isfinite(val[np.arange(M) != 5]))
    y_max = np.array([float(np.quantile(Y[0], 0.5)), np.inf])
    val, grad = mc_ei_value_grad(mu, var, dmu, dvar, eps, f, g, None, y_max, status=st)
    vref, gref = O.ei_value_grad(posts[0], Xs, np.ones(2), None, y_max)
    assert np.allclose(val, vref, rtol=1e-13, atol=0) and _grad_err(grad, gref) <= 1e-12
