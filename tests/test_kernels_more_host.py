"""CPU checks of the Matern12 (ExponentialKernel) and RationalQuadraticKernel reference maths and of the kernel-id
registry of the C ABI (which needs no device)."""
import ctypes
import math

import numpy as np
import pytest

from tests.kernels_more_oracle import KERNEL_MATERN12, KERNELS, RQ, O, kappa, kappa_dr_over_r, kernel_name, \
    mp_kappa_and_dr, adjudicator_mean_var_loglik
from tests.util_problems import make_problem

IDS = [kernel_name(k) for k in KERNELS]


@pytest.mark.parametrize("kernel", KERNELS, ids=IDS)
def test_kappa_against_mpmath(kernel):
    d2s = [1e-12, 1e-6, 0.01, 0.3, 1.0, 2.5, 7.0, 30.0, 200.0]
    for d2 in d2s:
        k_mp, dr_mp = mp_kappa_and_dr(d2, kernel)
        k, dr = float(kappa(d2, kernel)), float(kappa_dr_over_r(d2, kernel))
        # exp(-t) inherits t's rounding: a relative error of a few ulp times (1 + t)
        tol = 4e-16 * (1.0 + abs(math.log(k_mp)))
        assert abs(k - k_mp) <= tol * k_mp, (d2, k, k_mp)
        assert abs(dr - dr_mp) <= 10 * tol * abs(dr_mp), (d2, dr, dr_mp)
    assert float(kappa(0.0, kernel)) == 1.0


def test_r0_convention():
    # Matern12: kappa'(r)/r is unbounded as r -> 0 and defined as 0 at d2 == 0, with no NaN
    assert float(kappa_dr_over_r(0.0, KERNEL_MATERN12)) == 0.0
    assert np.isfinite(kappa_dr_over_r(np.array([0.0, 1e-300, 1e-30]), KERNEL_MATERN12)).all()
    # RQ: kappa'(r)/r -> -1 at r = 0, no convention needed
    for a in (0.5, 2.0, 50.0):
        assert float(kappa_dr_over_r(0.0, RQ(a))) == -1.0


def _dataset(n, d, seed, dup=False):
    X, Y, ls, amp, ns = make_problem(n, d, seed=seed)
    if dup:
        X[:, 1] = X[:, 0]
    return X, Y[0], ls[0], amp[0], ns[0]


@pytest.mark.parametrize("kernel", KERNELS, ids=IDS)
@pytest.mark.parametrize("dup", [False, True], ids=["plain", "duplicate"])
def test_loglik_grad_central_differences(kernel, dup):
    X, y, ls, amp, ns = _dataset(25, 3, seed=11, dup=dup)
    theta = np.concatenate([ls, [amp, ns]])
    ll, g = O.gp_loglik_grad(X, y, ls, amp, ns, kernel)
    assert np.isfinite(ll) and np.isfinite(g).all()
    assert ll == pytest.approx(O.gp_loglik(X, y, ls, amp, ns, kernel), rel=1e-12)
    for q in range(theta.size):
        h = 1e-6 * theta[q]
        tp, tm = theta.copy(), theta.copy()
        tp[q] += h
        tm[q] -= h
        fp = O.gp_loglik(X, y, tp[:3], tp[3], tp[4], kernel)
        fm = O.gp_loglik(X, y, tm[:3], tm[3], tm[4], kernel)
        fd = (fp - fm) / (2 * h)
        assert abs(g[q] - fd) <= 1e-5 * max(1.0, np.abs(g).max()), (q, g[q], fd)


@pytest.mark.parametrize("kernel", KERNELS, ids=IDS)
def test_mean_var_grad_central_differences(kernel):
    X, y, ls, amp, ns = _dataset(30, 3, seed=12)
    post = O.posterior_fit(X, y, ls, amp, ns, kernel)
    Xs = np.random.default_rng(5).random((3, 6))
    mu, var, dmu, dvar, st = O.mean_var_grad(post, Xs)
    assert (st == 0).all()
    for j in range(3):
        h = 1e-6
        P, M_ = Xs.copy(), Xs.copy()
        P[j] += h
        M_[j] -= h
        mp_, vp_ = O.mean_and_var(post, P)[:2]
        mm_, vm_ = O.mean_and_var(post, M_)[:2]
        np.testing.assert_allclose(dmu[j], (mp_ - mm_) / (2 * h), rtol=1e-5, atol=1e-6)
        np.testing.assert_allclose(dvar[j], (vp_ - vm_) / (2 * h), rtol=1e-5, atol=1e-6)


def test_matern12_candidate_on_training_point():
    """A candidate equal to a training point: that point contributes 0 to the x-gradient (symmetric subgradient)."""
    X, y, ls, amp, ns = _dataset(20, 2, seed=13)
    post = O.posterior_fit(X, y, ls, amp, ns, KERNEL_MATERN12)
    Xs = X[:, 3:4].copy()
    mu, var, dmu, dvar, st = O.mean_var_grad(post, Xs)
    assert np.isfinite(dmu).all() and np.isfinite(dvar).all()
    # the same sums without point 3
    keep = np.arange(20) != 3
    Xa, Xb = X / post.ls[:, None], Xs / post.ls[:, None]
    D2 = O._pairwise_sqdist_direct(Xa, Xb)[keep, 0]
    G = post.amp ** 2 * kappa_dr_over_r(D2, KERNEL_MATERN12)
    for j in range(2):
        diff = (Xb[j, 0] - Xa[j, keep]) / post.ls[j]
        assert dmu[j, 0] == pytest.approx(np.dot(post.alpha_w[keep], G * diff), rel=1e-12, abs=1e-12)


@pytest.mark.parametrize("kernel", KERNELS, ids=IDS)
def test_oracle_against_mpmath_adjudicator(kernel):
    X, y, ls, amp, ns = _dataset(12, 2, seed=14)
    Xs = np.random.default_rng(6).random((2, 4))
    post = O.posterior_fit(X, y, ls, amp, ns, kernel)
    mu, var = O.mean_and_var(post, Xs)[:2]
    mu_a, var_a, ll_a = adjudicator_mean_var_loglik(X, y, ls, amp, ns, kernel, Xs, dps=40)
    np.testing.assert_allclose(mu, mu_a, rtol=1e-10, atol=1e-12)
    np.testing.assert_allclose(var, var_a, rtol=1e-8, atol=1e-12)
    assert O.gp_loglik(X, y, ls, amp, ns, kernel) == pytest.approx(ll_a, rel=1e-11)


def _sk_gpr(kern, noise, X, y):
    from sklearn.gaussian_process import GaussianProcessRegressor
    g = GaussianProcessRegressor(kernel=kern, alpha=noise * noise, optimizer=None, normalize_y=False)
    return g.fit(X.T, y)


def test_oracle_against_sklearn_matern12_ard():
    pytest.importorskip("sklearn")
    from sklearn.gaussian_process.kernels import ConstantKernel, Matern
    X, y, ls, amp, ns = _dataset(40, 3, seed=15)
    lsc, ampc, nsc = O.condition_params(ls, amp, ns)
    kern = ConstantKernel(ampc * ampc, "fixed") * Matern(length_scale=lsc, length_scale_bounds="fixed", nu=0.5)
    K = O.kernel_matrix(X, None, lsc, ampc, KERNEL_MATERN12)
    np.testing.assert_allclose(K, kern(X.T), rtol=1e-13, atol=1e-15)
    Xs = np.random.default_rng(7).random((3, 20))
    m, s = _sk_gpr(kern, nsc, X, y).predict(Xs.T, return_std=True)
    mu, var = O.mean_and_var(O.posterior_fit(X, y, ls, amp, ns, KERNEL_MATERN12), Xs)[:2]
    np.testing.assert_allclose(mu, m, rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(var, s * s, rtol=1e-7, atol=1e-12)


@pytest.mark.parametrize("a", [0.5, 2.0, 50.0])
def test_oracle_against_sklearn_rq_isotropic(a):
    pytest.importorskip("sklearn")
    from sklearn.gaussian_process.kernels import ConstantKernel, RationalQuadratic
    X, y, _, amp, ns = _dataset(40, 3, seed=16)
    ls = np.full(3, 0.7)
    lsc, ampc, nsc = O.condition_params(ls, amp, ns)
    kern = ConstantKernel(ampc * ampc, "fixed") * RationalQuadratic(length_scale=lsc[0], alpha=a,
                                                                    length_scale_bounds="fixed", alpha_bounds="fixed")
    K = O.kernel_matrix(X, None, lsc, ampc, RQ(a))
    np.testing.assert_allclose(K, kern(X.T), rtol=1e-13, atol=1e-15)
    Xs = np.random.default_rng(8).random((3, 20))
    m, s = _sk_gpr(kern, nsc, X, y).predict(Xs.T, return_std=True)
    mu, var = O.mean_and_var(O.posterior_fit(X, y, ls, amp, ns, RQ(a)), Xs)[:2]
    np.testing.assert_allclose(mu, m, rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(var, s * s, rtol=1e-7, atol=1e-12)


def test_rq_large_a_tends_to_se():
    X, y, ls, amp, ns = _dataset(30, 3, seed=17)
    Xs = np.random.default_rng(9).random((3, 10))
    mu_rq, var_rq = O.mean_and_var(O.posterior_fit(X, y, ls, amp, ns, RQ(1e8)), Xs)[:2]
    mu_se, var_se = O.mean_and_var(O.posterior_fit(X, y, ls, amp, ns, O.KERNEL_SE), Xs)[:2]
    np.testing.assert_allclose(mu_rq, mu_se, rtol=1e-6, atol=1e-9)
    np.testing.assert_allclose(var_rq, var_se, rtol=1e-6, atol=1e-9)


# ---- the kernel-id registry of the C ABI: host-only, callable without boss_init ----

def _lib():
    import boss_b200  # noqa: F401
    from boss_b200 import _lib as L
    return L


def _register(L, a):
    out = ctypes.c_int(-1)
    rc = L.lib.boss_kernel_rational_quadratic(float(a), ctypes.byref(out))
    return rc, out.value


def test_registry_ids_without_init():
    L = _lib()
    assert L.KERNEL_MATERN12 == KERNEL_MATERN12
    rc1, id1 = _register(L, 2.0)
    rc2, id2 = _register(L, 2.0)
    rc3, id3 = _register(L, 0.75)
    assert rc1 == rc2 == rc3 == 0
    assert id1 == id2 and id1 != id3
    assert 256 <= id1 < 256 + L.RQ_SLOTS and 256 <= id3 < 256 + L.RQ_SLOTS
    assert L.kernel_rational_quadratic(2.0) == id1
    # the next double up is a different shape parameter and gets its own id
    rc4, id4 = _register(L, math.nextafter(2.0, 3.0))
    assert rc4 == 0 and id4 not in (id1, id3)


@pytest.mark.parametrize("a", [0.0, -0.0, -1.0, math.inf, -math.inf, math.nan])
def test_registry_rejects_bad_shape(a):
    L = _lib()
    rc, _ = _register(L, a)
    assert rc == -1   # BOSS_ERR_ARG
    assert "rq_a" in L.last_error()
    with pytest.raises(L.BossError):
        L.kernel_rational_quadratic(a)
