"""The host side of the Semiparametric theta-gradient (DESIGN.md 2.13) without a GPU: the numpy reference alpha^T J against
central differences of the oracle's log-likelihood, and the mirror's data_loglike_and_grad, theta box and gradient
OptimizationMAP fed the oracle's values in place of the library calls they make."""
import numpy as np
import pytest

from oracle import boss_oracle as O
from tests import loglik_mean_grad_oracle as MG


def _B():
    import boss_b200 as B
    return B


@pytest.fixture
def oracle_lib(monkeypatch):
    """The library calls of data_loglike / data_loglike_and_grad answered by the oracle."""
    from boss_b200 import _lib
    calls = {"mean": 0}

    def loglik_batch(X, Y, L, A, N, kernel_id=O.KERNEL_MATERN52, discrete_mask=None):
        return O.gp_loglik_batch(X, Y, L, A, N, kernel_id, discrete_mask)

    def loglik_grad_batch_mean(X, Y, J, L, A, N, kernel_id=O.KERNEL_MATERN52, discrete_mask=None):
        calls["mean"] += 1
        ll, gr = O.gp_loglik_grad_batch(X, Y, L, A, N, kernel_id, discrete_mask)
        _, gm = MG.gp_loglik_mean_grad_batch(X, Y, J, L, A, N, kernel_id, discrete_mask)
        return ll, gr, gm

    monkeypatch.setattr(_lib, "loglik_batch", loglik_batch)
    monkeypatch.setattr(_lib, "loglik_grad_batch_mean", loglik_grad_batch_mean)
    return calls


def _nonlinear_model(B, with_jacobian=True, kernel=None):
    """y_dim = 2, a mean nonlinear in theta, theta[1] pinned by a Dirac prior."""
    predict = lambda x, th: np.array([th[0] * np.sin(x[0]) + th[1] * x[1] ** 2,
                                      th[2] * np.exp(0.3 * x[0]) + th[1] * th[3] * x[1]])
    jac = lambda x, th: np.array([[np.sin(x[0]), x[1] ** 2, 0.0, 0.0],
                                  [0.0, th[3] * x[1], np.exp(0.3 * x[0]), th[1] * x[1]]])
    gp = B.GaussianProcess(kernel=kernel or B.Matern52Kernel(), lengthscale_priors=[B.mvlognormal([0, 0], [0.3, 0.3])] * 2,
                           amplitude_priors=[B.LogNormal()] * 2, noise_std_priors=[B.Dirac(0.1)] * 2)
    return B.Semiparametric(B.Parametric(predict, [B.Normal(), B.Dirac(0.7), B.Normal(), B.Normal()],
                                         jac if with_jacobian else None), gp)


def _nonlinear_data(B, n=24, seed=3):
    rng = np.random.default_rng(seed)
    X = rng.random((2, n)) * 3.0
    Y = np.stack([1.5 * np.sin(X[0]) + 0.7 * X[1] ** 2 + 0.2 * np.cos(3 * X[1]),
                  -0.5 * np.exp(0.3 * X[0]) + 0.7 * 1.2 * X[1] + 0.1 * np.sin(2 * X[0])])
    return B.ExperimentData(X, Y)


def linear_problem(B, n=30, seed=4, with_jacobian=True):
    """y = 2 x_1 + 0.5 + a smooth residual; Parametric theta_1 x_1 + theta_2 (Jacobian [x_1, 1])."""
    rng = np.random.default_rng(seed)
    X = rng.random((2, n)) * 4.0
    Y = (2.0 * X[0] + 0.5 + 0.3 * np.sin(2.0 * X[1]))[None, :]
    gp = B.GaussianProcess(kernel=B.Matern52Kernel(), lengthscale_priors=[B.mvlognormal([0, 0], [0.5, 0.5])],
                           amplitude_priors=[B.LogNormal()], noise_std_priors=[B.Dirac(0.05)])
    jac = (lambda x, th: np.array([[x[0], 1.0]])) if with_jacobian else None
    model = B.Semiparametric(B.Parametric(lambda x, th: np.array([th[0] * x[0] + th[1]]),
                                          [B.Uniform(-3, 3), B.Uniform(-1, 1)], jac), gp)
    return B.BossProblem(lambda x: x, B.Domain(([0.0, 0.0], [4.0, 4.0])), B.ExpectedImprovement(B.LinFitness([1.0])),
                         model, B.ExperimentData(X, Y))


@pytest.mark.parametrize("kernel_id", [O.KERNEL_SE, O.KERNEL_MATERN32, O.KERNEL_MATERN52])
def test_reference_matches_central_differences_of_the_loglik(kernel_id):
    """alpha^T J is d/dtheta of gp_loglik(X, y - m(X; theta)) for a mean nonlinear in theta, discrete dimension 1."""
    rng = np.random.default_rng(kernel_id)
    X = rng.random((3, 40)) * 2.0
    X[1] = np.round(X[1] * 2.0)
    mask = np.array([0, 1, 0], dtype=np.uint8)
    y = np.sin(2 * X[0]) + 0.5 * X[1] + 0.1 * X[2]
    m = lambda th: th[0] * np.sin(2 * X[0]) + np.exp(th[1] * X[2]) + th[2] * th[0] * X[1]
    J = lambda th: np.stack([np.sin(2 * X[0]) + th[2] * X[1], X[2] * np.exp(th[1] * X[2]), th[0] * X[1]])
    th = np.array([0.8, -0.3, 0.4])
    ls, amp, ns = np.array([0.7, 1.3, 0.9]), 1.1, 0.1
    ll, g = MG.gp_loglik_mean_grad(X, y - m(th), J(th), ls, amp, ns, kernel_id, mask)
    assert ll == O.gp_loglik(X, y - m(th), ls, amp, ns, kernel_id, mask)
    h = 1e-6
    for c in range(3):
        tp, tm = th.copy(), th.copy()
        tp[c] += h; tm[c] -= h
        fd = (O.gp_loglik(X, y - m(tp), ls, amp, ns, kernel_id, mask) - O.gp_loglik(X, y - m(tm), ls, amp, ns, kernel_id, mask)) / (2 * h)
        assert abs(g[c] - fd) <= 1e-6 * max(1.0, abs(fd)), (c, g[c], fd)


def test_data_loglike_and_grad_of_a_semiparametric_model(oracle_lib):
    """Two output slices, theta-gradient summed over them, against central differences of data_loglike in every theta
    entry; the GP part against the oracle's hyper-parameter gradient; one library call per slice for a list."""
    B = _B()
    model, data = _nonlinear_model(B), _nonlinear_data(B)
    p = B.SemiparametricParams(np.array([1.2, 0.7, -0.4, 0.9]), np.array([[0.8, 1.1], [1.3, 0.6]]), np.array([1.0, 0.7]),
                               np.array([0.1, 0.1]))
    ll = B.data_loglike(model, data)
    v, g = B.data_loglike_and_grad(model, data)(p)
    assert abs(v - ll(p)) <= 1e-12 * abs(v)
    assert isinstance(g, B.SemiparametricParams) and g.theta.shape == (4,)
    h = 1e-6
    for c in range(4):
        tp, tm = p.theta.copy(), p.theta.copy()
        tp[c] += h; tm[c] -= h
        fd = (ll(B.SemiparametricParams(tp, p.lengthscales, p.amplitudes, p.noise_std))
              - ll(B.SemiparametricParams(tm, p.lengthscales, p.amplitudes, p.noise_std))) / (2 * h)
        assert abs(g.theta[c] - fd) <= 1e-6 * max(1.0, abs(fd)), (c, g.theta[c], fd)
    for i in range(2):
        mean_i = np.array([model.parametric.predict(data.X[:, j], p.theta)[i] for j in range(data.X.shape[1])])
        _, gr = O.gp_loglik_grad(data.X, data.Y[i] - mean_i, p.lengthscales[:, i], p.amplitudes[i], p.noise_std[i],
                                 O.KERNEL_MATERN52)
        assert np.array_equal(g.lengthscales[:, i], gr[:2]) and g.amplitudes[i] == gr[2] and g.noise_std[i] == gr[3]
    oracle_lib["mean"] = 0
    vals, grads = B.data_loglike_and_grad(model, data)([p, p, p])
    assert oracle_lib["mean"] == 2
    assert np.all(vals == v) and all(np.array_equal(q.theta, g.theta) for q in grads)


def test_without_jacobian_the_theta_gradient_is_not_available():
    B = _B()
    with pytest.raises(NotImplementedError):
        B.data_loglike_and_grad(_nonlinear_model(B, with_jacobian=False), _nonlinear_data(B))


def test_search_box():
    """theta: [min - 30, max + 30] over the starts, cut to a Uniform prior's support; log-parameters: [-30, 30]."""
    B = _B()
    from boss_b200.model_fitters import _search_box
    V0 = np.array([[0.5, -0.2, 0.1, 0.2, 0.0, -2.3], [-1.5, 0.6, 0.3, -0.1, 0.4, -2.3]])     # theta (2) | log lambda, alpha, sigma
    lo, hi = _search_box(linear_problem(B).model, V0)
    assert np.array_equal(lo, [-3.0, -1.0, -30, -30, -30, -30]) and np.array_equal(hi, [3.0, 1.0, 30, 30, 30, 30])
    model = _nonlinear_model(B)                                                                 # Normal / Dirac priors
    V0 = np.array([[1.0, 0.7, -40.0, 2.0] + [0.0] * 8, [3.0, 0.7, -41.0, -2.0] + [0.0] * 8])
    lo, hi = _search_box(model, V0)
    assert np.array_equal(lo[:4], [-29.0, -29.3, -71.0, -32.0]) and np.array_equal(hi[:4], [33.0, 30.7, -10.0, 32.0])
    assert np.all(lo[4:] == -30.0) and np.all(hi[4:] == 30.0)
    gp = _problem_gp(B)
    lo, hi = _search_box(gp, np.zeros((3, 5)))
    assert np.all(lo == -30.0) and np.all(hi == 30.0)


def _problem_gp(B):
    return B.GaussianProcess(lengthscale_priors=[B.mvlognormal([0, 0], [1, 1])], amplitude_priors=[B.LogNormal()],
                             noise_std_priors=[B.Dirac(0.1)])


def test_gradient_optimization_map_of_a_semiparametric_model(oracle_lib):
    """Gradient OptimizationMAP on the oracle's values: reaches the compass search's log-likelihood, reports the value
    at its point, keeps Dirac-pinned entries exact; without a Jacobian "lbfgs" is the compass search, bit for bit."""
    B = _B()
    prob = linear_problem(B)
    ll = B.model_loglike(prob.model, prob.data)
    grad = B.estimate_parameters(B.OptimizationMAP(multistart=6, iters=30, seed=21, algorithm="lbfgs"), prob)
    comp = B.estimate_parameters(B.OptimizationMAP(multistart=6, iters=30, seed=21, algorithm="compass"), prob)
    assert oracle_lib["mean"] > 0
    for r in (grad, comp):
        assert abs(ll(r.params) - r.loglike) <= 1e-8 * abs(r.loglike)
        assert np.all(r.params.noise_std == 0.05)
    assert grad.loglike >= comp.loglike - 0.05 * abs(comp.loglike)
    assert abs(grad.params.theta[0] - 2.0) < 0.3
    nj = linear_problem(B, with_jacobian=False)
    a = B.estimate_parameters(B.OptimizationMAP(multistart=4, iters=8, seed=5, algorithm="lbfgs"), nj)
    b = B.estimate_parameters(B.OptimizationMAP(multistart=4, iters=8, seed=5, algorithm="compass"), nj)
    assert a.loglike == b.loglike and np.array_equal(a.params.theta, b.params.theta)
    assert np.array_equal(a.params.lengthscales, b.params.lengthscales) and np.array_equal(a.params.amplitudes, b.params.amplitudes)
    # theta[1] pinned by a Dirac prior stays exact through the gradient search
    model, data = _nonlinear_model(B), _nonlinear_data(B, n=16)
    pb = B.BossProblem(lambda x: x, B.Domain(([0.0, 0.0], [3.0, 3.0])), B.ExpectedImprovement(B.LinFitness([1.0, 0.0])),
                       model, data)
    r = B.estimate_parameters(B.OptimizationMAP(multistart=3, iters=10, seed=2, algorithm="lbfgs"), pb)
    assert r.params.theta[1] == 0.7 and np.isfinite(r.loglike)
