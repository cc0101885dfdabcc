"""GPU parity tests: the CUDA path through the C ABI vs the CPU oracle on identical seeded inputs.

Tolerances are the north star's: relative error <= 1e-9 for posterior mean / variance / EI,
<= 1e-8 for the log marginal likelihood, argmax index exact on tie-free candidate sets.
"""
import numpy as np
import pytest

from oracle import boss_oracle as O
from tests.util_problems import make_hyper_samples, make_problem, relerr

pytestmark = pytest.mark.gpu

TOL_POST = 1e-9
TOL_LL = 1e-8


# ---------------------------------------------------------------------------------------------
# the FP64 tensor-core mainloop in isolation
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("M,N,K", [(128, 128, 16), (128, 128, 80), (256, 384, 160), (130, 70, 33), (512, 128, 2048)])
def test_gemm_core(lib, M, N, K):
    rng = np.random.default_rng(M * 7 + N * 3 + K)
    A = rng.standard_normal((M, K)); B = rng.standard_normal((N, K))
    C = lib.dbg_gemm_nt(A, B)
    ref = A @ B.T
    assert np.max(np.abs(C - ref)) <= 1e-12 * K


# ---------------------------------------------------------------------------------------------
# fit: kernel matrix + blocked Cholesky + triangular inverse + alpha + loglik
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,d,kid", [(3, 2, 2), (20, 2, 0), (128, 1, 1), (200, 6, 2), (300, 3, 0), (512, 6, 2),
                                     (640, 10, 1)])
def test_fit_factors(lib, n, d, kid):
    X, Y, ls, amp, ns = make_problem(n, d, seed=100 + n)
    gp = lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], kid)
    assert gp is not None
    post = O.posterior_fit(X, Y[0], ls[0], amp[0], ns[0], kid)
    L, W, alpha = lib.dbg_factors(gp)
    Lref = post.U.T
    assert np.max(np.abs(L - Lref)) / np.max(np.abs(Lref)) < 1e-11
    Wref = np.linalg.inv(Lref)
    assert np.max(np.abs(W - Wref)) / np.max(np.abs(Wref)) < 1e-9
    assert np.max(np.abs(alpha - post.alpha_w)) / np.max(np.abs(post.alpha_w)) < 1e-9
    ll = O.gp_loglik(X, Y[0], ls[0], amp[0], ns[0], kid)
    assert abs(gp.loglik - ll) <= TOL_LL * abs(ll)
    gp.free()


# ---------------------------------------------------------------------------------------------
# predict (mean_and_var) incl. prior mean, vector == matrix API, clip
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,d,kid,M", [(3, 2, 2, 7), (20, 2, 0, 300), (200, 6, 2, 1000), (512, 8, 1, 777),
                                       (1024, 10, 2, 2048)])
def test_predict(lib, n, d, kid, M):
    X, Y, ls, amp, ns = make_problem(n, d, seed=200 + n)
    rng = np.random.default_rng(n + M)
    Xs = rng.random((d, M))
    pm = rng.standard_normal(M)
    gp = lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], kid)
    post = O.posterior_fit(X, Y[0], ls[0], amp[0], ns[0], kid)
    mu_ref, var_ref, st_ref = O.mean_and_var(post, Xs, pm)
    mu, var, st = lib.gp_predict(gp, Xs, pm)
    assert np.array_equal(st, st_ref)
    assert relerr(mu, mu_ref) <= TOL_POST, relerr(mu, mu_ref)
    assert relerr(var, var_ref) <= TOL_POST, relerr(var, var_ref)
    # vector API == column of the matrix API  (test/unit/test/models/gaussian_process.jl:115-126)
    m1, v1, _ = lib.gp_predict(gp, Xs[:, 3], pm[3:4])
    assert m1[0] == mu[3] and v1[0] == var[3]
    gp.free()


def test_predict_at_training_points_interpolates(lib):
    X, Y, ls, amp, ns = make_problem(40, 2, seed=5, noise=1e-3)
    gp = lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], 2)
    mu, var, st = lib.gp_predict(gp, X)
    assert np.allclose(mu, Y[0], atol=0.01)
    assert np.all(st == 0) and np.all(var >= 0)
    far = np.full((2, 1), 1000.0)
    mu_f, var_f, _ = lib.gp_predict(gp, far)
    assert abs(mu_f[0]) < 1e-8 and abs(var_f[0] - (1.0 + 1e-8) ** 2) < 1e-8
    gp.free()


def test_discrete_kernel(lib):
    X, Y, ls, amp, ns = make_problem(60, 3, seed=9)
    X = X * 6.0
    mask = np.array([True, False, True])
    rng = np.random.default_rng(2)
    Xs = rng.random((3, 257)) * 6.0
    gp = lib.gp_fit(X, Y[0], ls[0] * 3, amp[0], ns[0], 1, mask)
    post = O.posterior_fit(X, Y[0], ls[0] * 3, amp[0], ns[0], 1, mask)
    mu_ref, var_ref, _ = O.mean_and_var(post, Xs)
    mu, var, _ = lib.gp_predict(gp, Xs)
    assert relerr(mu, mu_ref) <= TOL_POST and relerr(var, var_ref) <= TOL_POST
    gp.free()


# ---------------------------------------------------------------------------------------------
# acquisition: EI, EI x PoF, PoF only, nothing; bounds / cons guards; BI average; argmax
# ---------------------------------------------------------------------------------------------
def _fit_all(lib, X, Y, ls, amp, ns, kid):
    gps = [lib.gp_fit(X, Y[i], ls[i], amp[i], ns[i], kid) for i in range(Y.shape[0])]
    posts = [O.posterior_fit(X, Y[i], ls[i], amp[i], ns[i], kid) for i in range(Y.shape[0])]
    return gps, posts


def _ei_mask(acq_ref):
    # relative comparison where EI is representable without extreme-tail amplification
    return acq_ref > 1e-200


@pytest.mark.parametrize("case", ["ei", "ei_pof", "pof", "none"])
def test_ei_score_cases(lib, case):
    n, d, y_dim, M = 300, 4, 3, 5000
    X, Y, ls, amp, ns = make_problem(n, d, seed=31, y_dim=y_dim)
    gps, posts = _fit_all(lib, X, Y, ls, amp, ns, 2)
    rng = np.random.default_rng(77)
    Xs = rng.random((d, M)) * 1.2 - 0.1           # some candidates out of bounds
    lb, ub = np.zeros(d), np.ones(d)
    cons = (rng.random(M) > 0.1).astype(np.uint8)
    coefs = np.array([1.0, 0.0, 0.25])
    y_max = np.array([np.inf, float(np.quantile(Y[1], 0.7)), float(np.quantile(Y[2], 0.7))])
    best = O.best_so_far(coefs, Y, y_max)
    kw = dict(ei=(best, None), ei_pof=(best, y_max), pof=(None, y_max), none=(None, None))[case]
    acq_ref, _, _ = O.ei_acquisition([posts], Xs, coefs, kw[0], kw[1], lb, ub, cons)
    acq, bv, bi = lib.ei_score(gps, y_dim, 1, Xs, coefs, kw[0], kw[1], lb, ub, cons)
    mask = _ei_mask(acq_ref)
    assert relerr(acq[mask], acq_ref[mask]) <= TOL_POST, relerr(acq[mask], acq_ref[mask])
    assert np.all(acq[~mask] <= 1e-200)
    assert np.all(acq[(cons == 0) | ~O.in_bounds(Xs, lb, ub)] == 0.0)
    assert bi == O.julia_argmax_fast(acq_ref)
    assert bv == acq[bi]
    for g in gps:
        g.free()


def test_ei_bi_sample_average(lib):
    n, d, M, S = 150, 3, 1500, 4
    X, Y, _, _, _ = make_problem(n, d, seed=41)
    L, A, N = make_hyper_samples(S, d, seed=42)
    gps = [lib.gp_fit(X, Y[0], L[s], A[s], N[s], 0) for s in range(S)]
    posts = [[O.posterior_fit(X, Y[0], L[s], A[s], N[s], 0)] for s in range(S)]
    Xs = np.random.default_rng(1).random((d, M))
    best = float(np.median(Y[0]))
    acq_ref, _, _ = O.ei_acquisition(posts, Xs, [1.0], best, None)
    acq, bv, bi = lib.ei_score(gps, 1, S, Xs, [1.0], best, None)
    assert relerr(acq, acq_ref) <= TOL_POST
    assert bi == O.julia_argmax_fast(acq_ref)
    for g in gps:
        g.free()


def test_ei_known_answers_on_device(lib):
    """Reference EI known answers pushed through the device epilogue: a GP with a far-away single
    training point has mu = prior mean, var = a^2, so EI follows the closed form exactly."""
    X = np.array([[1000.0]]); y = np.array([0.0])
    gp = lib.gp_fit(X, y, [1.0], 1.0, 0.1, 0)
    Xs = np.zeros((1, 4))
    acq, _, _ = lib.ei_score([gp], 1, 1, Xs, [1.0], 0.0, None, prior_mean_s=np.array([[0.0, -10.0, 1.0, 0.5]]))
    a2 = (1.0 + 1e-8) ** 2
    ref = O.expected_improvement([1.0], np.array([[0.0, -10.0, 1.0, 0.5]]), np.full((1, 4), a2 + 1e-18), 0.0)
    assert relerr(acq, ref) <= 1e-10     # z = -10 tail: erfc ulp differences are amplified ~|z|^2
    assert acq[1] < 1e-20
    gp.free()


def test_argmax_first_max_and_ties(lib):
    X, Y, ls, amp, ns = make_problem(50, 2, seed=3)
    gp = lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], 2)
    rng = np.random.default_rng(0)
    base = rng.random((2, 700))
    Xs = np.concatenate([base, base[:, ::-1]], axis=1)     # every candidate appears twice
    acq, bv, bi = lib.ei_score([gp], 1, 1, Xs, [1.0], float(np.median(Y[0])), None)
    assert bi == int(np.argmax(acq))                       # first maximal element
    # everything out of bounds -> all zeros -> index 0
    acq0, bv0, bi0 = lib.ei_score([gp], 1, 1, Xs + 5.0, [1.0], 0.0, None, np.zeros(2), np.ones(2))
    assert np.all(acq0 == 0.0) and bi0 == 0 and bv0 == 0.0
    gp.free()


# ---------------------------------------------------------------------------------------------
# batched log marginal likelihood
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,d,kid,S", [(3, 2, 2, 5), (20, 2, 0, 33), (130, 3, 1, 17), (512, 6, 2, 24), (512, 6, 0, 8),
                                       (1024, 8, 2, 4)])
def test_loglik_batch(lib, n, d, kid, S):
    X, Y, _, _, _ = make_problem(n, d, seed=300 + n)
    L, A, N = make_hyper_samples(S, d, seed=301 + n)
    ref = O.gp_loglik_batch(X, Y[0], L, A, N, kid)
    out = lib.loglik_batch(X, Y[0], L, A, N, kid)
    assert relerr(out, ref) <= TOL_LL, relerr(out, ref)


def test_loglik_batch_per_sample_mean(lib):
    """Semiparametric: y - m_theta(X) differs per sample (src/models/semiparametric.jl:86-92)."""
    n, d, S = 100, 2, 6
    X, Y, _, _, _ = make_problem(n, d, seed=8)
    L, A, N = make_hyper_samples(S, d, seed=9)
    theta = np.random.default_rng(3).standard_normal((S, 2))
    Ymm = np.stack([Y[0] - (theta[s, 0] * X[0] + theta[s, 1]) for s in range(S)])
    ref = O.gp_loglik_batch(X, Ymm, L, A, N, 2)
    out = lib.loglik_batch(X, Ymm, L, A, N, 2)
    assert relerr(out, ref) <= TOL_LL


def test_not_positive_definite(lib):
    X = np.zeros((1, 40)); y = np.arange(40.0)
    # zero noise, 40 identical points: K = a^2 * ones is numerically singular -> some pivot is <= 0
    out = lib.loglik_batch(X, y, np.array([[1.0], [1.0]]), np.array([1e6, 1.0]), np.array([0.0, 0.5]), 0)
    assert out[0] == -np.inf and np.isfinite(out[1])
    assert O.gp_loglik(X, y, [1.0], 1e6, 0.0, 0) == -np.inf
    assert lib.gp_fit(X, y, [1.0], 1e6, 0.0, 0) is None


def test_negative_hyperparameters_rejected(lib):
    X, Y, ls, amp, ns = make_problem(10, 2, seed=1)
    with pytest.raises(lib.BossError):
        lib.gp_fit(X, Y[0], -ls[0], amp[0], ns[0], 2)


# ---------------------------------------------------------------------------------------------
# headline shape: n = 2048, d = 8, Matern52 (BASELINE.json configs[1]) on a 65 536-candidate subset
# ---------------------------------------------------------------------------------------------
def test_headline_shape_parity(lib):
    n, d, M = 2048, 8, 65536
    X, Y, ls, amp, ns = make_problem(n, d, seed=1002)
    Xs = np.random.default_rng(2002).random((d, M))
    gp = lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], 2)
    post = O.posterior_fit(X, Y[0], ls[0], amp[0], ns[0], 2)
    ll = O.gp_loglik(X, Y[0], ls[0], amp[0], ns[0], 2)
    assert abs(gp.loglik - ll) <= TOL_LL * abs(ll)
    mu_ref, var_ref, st_ref = O.mean_and_var(post, Xs)
    mu, var, st = lib.gp_predict(gp, Xs)
    assert relerr(mu, mu_ref) <= TOL_POST and relerr(var, var_ref) <= TOL_POST
    best = float(np.max(Y[0]))
    acq_ref, _, _ = O.ei_acquisition([[post]], Xs, [1.0], best, None)
    acq, bv, bi = lib.ei_score([gp], 1, 1, Xs, [1.0], best, None)
    mask = _ei_mask(acq_ref)
    assert relerr(acq[mask], acq_ref[mask]) <= TOL_POST
    assert bi == O.julia_argmax_fast(acq_ref)
    # size-independent property: scoring a permutation permutes the scores bit-exactly
    perm = np.random.default_rng(0).permutation(M)
    acq_p, _, bi_p = lib.ei_score([gp], 1, 1, Xs[:, perm], [1.0], best, None)
    assert np.array_equal(acq_p, acq[perm])
    gp.free()


# ---------------------------------------------------------------------------------------------
# analytic x-gradients (multi-start optimiser path, config C4 style)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kid,d,n", [(2, 4, 300), (0, 3, 130), (1, 2, 64)])
def test_ei_value_grad_single_output(lib, kid, d, n):
    X, Y, ls, amp, ns = make_problem(n, d, seed=500 + n)
    gp = lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], kid)
    post = O.posterior_fit(X, Y[0], ls[0], amp[0], ns[0], kid)
    Xs = np.random.default_rng(4).random((d, 700))
    best = float(np.quantile(Y[0], 0.8))
    val_ref, grad_ref = O.ei_value_grad([post], Xs, [1.0], best, None)
    val, grad = lib.ei_value_grad([gp], 1, 1, Xs, [1.0], best, None)
    assert relerr(val, val_ref) <= TOL_POST
    scale = np.max(np.abs(grad_ref), axis=1, keepdims=True)
    assert np.max(np.abs(grad - grad_ref) / scale) <= 1e-8
    # value path unchanged by gradient mode
    acq, _, _ = lib.ei_score([gp], 1, 1, Xs, [1.0], best, None)
    assert np.array_equal(acq, val)
    gp.free()


def test_ei_value_grad_multi_output_pof_and_prior_mean(lib):
    n, d, y_dim, M = 200, 3, 2, 400
    X, Y, ls, amp, ns = make_problem(n, d, seed=61, y_dim=y_dim)
    theta = np.array([0.3, -0.2, 0.1])
    mean_X = theta @ X                                  # Semiparametric: linear parametric mean on output 0
    Ymm = Y.copy(); Ymm[0] -= mean_X
    gps = [lib.gp_fit(X, Ymm[i], ls[i], amp[i], ns[i], 2) for i in range(y_dim)]
    posts = [O.posterior_fit(X, Ymm[i], ls[i], amp[i], ns[i], 2) for i in range(y_dim)]
    Xs = np.random.default_rng(5).random((d, M))
    pm = np.stack([theta @ Xs, np.zeros(M)])
    pmg = np.zeros((y_dim, d, M)); pmg[0] = theta[:, None]
    coefs = [1.0, 0.2]; y_max = [np.inf, float(np.quantile(Y[1], 0.6))]
    best = float(np.median(np.asarray(coefs) @ Y))
    val, grad = lib.ei_value_grad(gps, y_dim, 1, Xs, coefs, best, y_max, prior_mean_s=pm, prior_mean_grad_s=pmg)
    ref, _, _ = O.ei_acquisition([posts], Xs, coefs, best, y_max, prior_mean_s=pm)
    assert relerr(val, ref) <= TOL_POST
    # central finite differences of the oracle acquisition (prior mean moves with x)
    h = 1e-6
    for j in range(d):
        Xp = Xs.copy(); Xp[j] += h
        Xm = Xs.copy(); Xm[j] -= h
        fp, _, _ = O.ei_acquisition([posts], Xp, coefs, best, y_max, prior_mean_s=np.stack([theta @ Xp, np.zeros(M)]))
        fm, _, _ = O.ei_acquisition([posts], Xm, coefs, best, y_max, prior_mean_s=np.stack([theta @ Xm, np.zeros(M)]))
        fd = (fp - fm) / (2 * h)
        assert np.allclose(grad[j], fd, rtol=5e-5, atol=1e-8), j
    for g in gps:
        g.free()


def test_ei_value_grad_guards(lib):
    X, Y, ls, amp, ns = make_problem(80, 2, seed=71)
    gp = lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], 2)
    Xs = np.array([[0.5, 1.5, 0.2], [0.5, 0.5, -0.1]])
    val, grad = lib.ei_value_grad([gp], 1, 1, Xs, [1.0], float(np.median(Y[0])), None, np.zeros(2), np.ones(2))
    assert val[1] == 0.0 and val[2] == 0.0 and np.all(grad[:, 1:] == 0.0)
    assert val[0] > 0.0 and np.any(grad[:, 0] != 0.0)
    gp.free()


def test_small_batch_split_is_bitwise_invariant(lib):
    """Small candidate batches are dealt to several CTAs per candidate block (row-block / training-chunk
    splits).  Partial sums are kept per row block and added in a fixed order, so the same point scores
    bit-identically whether it arrives alone, in a 1 000-start batch or inside a 40 000-candidate grid
    (=> results do not depend on how a batch is sharded over GPUs)."""
    n, d = 700, 4
    X, Y, ls, amp, ns = make_problem(n, d, seed=91)
    gp = lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], 2)
    post = O.posterior_fit(X, Y[0], ls[0], amp[0], ns[0], 2)
    rng = np.random.default_rng(92)
    big = rng.random((d, 40000))                       # 313 candidate blocks: unsplit
    best = float(np.quantile(Y[0], 0.9))
    acq_big, _, _ = lib.ei_score([gp], 1, 1, big, [1.0], best, None)
    for m in (1, 100, 1000):                           # 1 / 1 / 8 candidate blocks: split over CTAs
        acq_s, _, bi = lib.ei_score([gp], 1, 1, big[:, :m], [1.0], best, None)
        assert np.array_equal(acq_s, acq_big[:m])
        assert bi == int(np.argmax(acq_big[:m]))
        val, grad = lib.ei_value_grad([gp], 1, 1, big[:, :m], [1.0], best, None)
        assert np.array_equal(val, acq_big[:m])
    val_big, grad_big = lib.ei_value_grad([gp], 1, 1, big[:, :38000], [1.0], best, None)
    val_s, grad_s = lib.ei_value_grad([gp], 1, 1, big[:, :1000], [1.0], best, None)
    assert np.array_equal(grad_s, grad_big[:, :1000])
    ref, gref = O.ei_value_grad([post], big[:, :1000], [1.0], best, None)
    assert relerr(val_s, ref) <= TOL_POST
    assert np.max(np.abs(grad_s - gref) / np.max(np.abs(gref), axis=1, keepdims=True)) <= 1e-8
    gp.free()


@pytest.mark.parametrize("n,d,kid,M", [(60, 2, 2, 5), (300, 4, 0, 200), (700, 3, 1, 333)])
def test_posterior_cov(lib, n, d, kid, M):
    """cov / mean_and_cov(::GaussianProcessPosterior, X) (gaussian_process.jl:163-167,180-184)."""
    X, Y, ls, amp, ns = make_problem(n, d, seed=600 + n)
    gp = lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], kid)
    post = O.posterior_fit(X, Y[0], ls[0], amp[0], ns[0], kid)
    Xs = np.random.default_rng(6).random((d, M))
    pm = np.linspace(-1, 1, M)
    mu, cov, rc = lib.gp_cov(gp, Xs, prior_mean_s=pm)
    C_ref, st = O.posterior_cov(post, Xs)
    mu_ref, var_ref, _ = O.mean_and_var(post, Xs, pm)
    assert rc == 0 and not st.any()
    assert relerr(mu, mu_ref) <= TOL_POST
    assert relerr(np.diag(cov), var_ref) <= TOL_POST
    # off-diagonal entries cancel to ~0 between distant points: compare relative to sqrt(var_i var_j)
    scale = np.sqrt(np.outer(var_ref, var_ref))
    assert np.max(np.abs(cov - C_ref) / scale) <= TOL_POST
    assert np.array_equal(cov, cov.T)
    # the diagonal agrees with the variance path (different summation order: V^T V tile product vs fused squares)
    _, var, _ = lib.gp_predict(gp, Xs)
    assert relerr(np.diag(cov), var) <= 1e-11
    gp.free()


# ---------------------------------------------------------------------------------------------
# warp-register small-n log-likelihood path (n <= 32, csrc/small.cuh)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,d,kid,S", [(1, 1, 2, 3), (2, 3, 0, 9), (17, 5, 1, 100), (30, 2, 0, 1000), (32, 9, 2, 257),
                                       (33, 2, 2, 40)])
def test_loglik_small_n_warp_path(lib, n, d, kid, S):
    X, Y, _, _, _ = make_problem(n, d, seed=700 + n)
    L, A, N = make_hyper_samples(S, d, seed=701 + n)
    ref = O.gp_loglik_batch(X, Y[0], L, A, N, kid)
    out = lib.loglik_batch(X, Y[0], L, A, N, kid)
    assert relerr(out, ref) <= TOL_LL, relerr(out, ref)
    # the blocked (128-padded) factorisation used by boss_gp_fit agrees with the warp path
    for s in range(min(S, 3)):
        gp = lib.gp_fit(X, Y[0], L[s], A[s], N[s], kid)
        assert abs(gp.loglik - out[s]) <= 1e-11 * abs(out[s])
        gp.free()


def test_loglik_small_n_discrete_mean_and_failures(lib):
    n, d, S = 24, 3, 12
    X, Y, _, _, _ = make_problem(n, d, seed=801)
    X = X * 4.0
    mask = np.array([True, False, True])
    L, A, N = make_hyper_samples(S, d, seed=802)
    Ymm = Y[0][None, :] - np.linspace(-1, 1, S)[:, None]
    ref = O.gp_loglik_batch(X, Ymm, L, A, N, 2, discrete_mask=mask)
    out = lib.loglik_batch(X, Ymm, L, A, N, 2, discrete_mask=mask)
    assert relerr(out, ref) <= TOL_LL
    # 24 identical points, zero noise, huge amplitude: K = a^2 * ones is numerically singular -> -Inf for that sample only
    Xz = np.zeros((1, 24)); yz = np.arange(24.0)
    out = lib.loglik_batch(Xz, yz, np.array([[1.0], [1.0]]), np.array([1e6, 1.0]), np.array([0.0, 0.5]), 0)
    assert out[0] == -np.inf and np.isfinite(out[1])
    assert abs(out[1] - O.gp_loglik(Xz, yz, [1.0], 1.0, 0.5, 0)) <= TOL_LL * abs(out[1])
    with pytest.raises(lib.BossError):
        lib.loglik_batch(X, Y[0], -L, A, N, 2)


# ---------------------------------------------------------------------------------------------
# incremental factor cache: boss_gp_append (SequentialBatchAM speculative points, BO iterations)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n0,m,d,kid", [(5, 40, 2, 2), (120, 20, 3, 0), (250, 10, 4, 1)])
def test_append_matches_full_refit(lib, n0, m, d, kid):
    """Appending points one at a time == fitting all of them at once (crosses the 128-block capacity boundary:
    the handle is repacked to a larger P-layout)."""
    n = n0 + m
    X, Y, ls, amp, ns = make_problem(n, d, seed=900 + n0)
    gp = lib.gp_fit(X[:, :n0], Y[0, :n0], ls[0], amp[0], ns[0], kid)
    for k in range(n0, n):
        assert lib.gp_append(gp, X[:, k], Y[0, k])
    assert gp.n == n
    post = O.posterior_fit(X, Y[0], ls[0], amp[0], ns[0], kid)
    ll = O.gp_loglik(X, Y[0], ls[0], amp[0], ns[0], kid)
    assert abs(gp.loglik - ll) <= TOL_LL * abs(ll)
    L, W, al = lib.dbg_factors(gp)
    assert np.max(np.abs(L - post.U.T)) <= 1e-10 * np.max(np.abs(post.U))
    assert relerr(al, post.alpha_w) <= 1e-8
    Xs = np.random.default_rng(3).random((d, 500))
    mu, var, st = lib.gp_predict(gp, Xs)
    mu_r, var_r, _ = O.mean_and_var(post, Xs)
    assert relerr(mu, mu_r) <= TOL_POST and relerr(var, var_r) <= TOL_POST
    best = float(np.quantile(Y[0], 0.8))
    acq, _, bi = lib.ei_score([gp], 1, 1, Xs, [1.0], best, None)
    ref, _, _ = O.ei_acquisition([[post]], Xs, [1.0], best, None)
    mask = _ei_mask(ref)
    assert relerr(acq[mask], ref[mask]) <= TOL_POST and bi == O.julia_argmax_fast(ref)
    gp.free()


def test_append_duplicate_point_without_noise_is_rejected(lib):
    X, Y, ls, amp, ns = make_problem(30, 2, seed=5)
    gp = lib.gp_fit(X, Y[0], ls[0], 1e6, 0.0, 0)       # huge amplitude, zero noise: a repeated point is singular
    ll0 = gp.loglik
    ok = lib.gp_append(gp, X[:, 3], Y[0, 3])
    if not ok:                                          # rejected: handle unchanged
        assert gp.n == 30 and gp.loglik == ll0
        mu, var, _ = lib.gp_predict(gp, X[:, :5])
        assert np.all(np.isfinite(mu))
    gp.free()


# ---------------------------------------------------------------------------------------------
# hyper-parameter gradient of the log marginal likelihood (SURVEY.md 8f rank 2)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,d,kid,S", [(3, 2, 2, 4), (20, 2, 0, 9), (130, 3, 1, 7), (300, 5, 2, 6), (512, 6, 0, 5)])
def test_loglik_grad_batch(lib, n, d, kid, S):
    X, Y, _, _, _ = make_problem(n, d, seed=1300 + n)
    L, A, N = make_hyper_samples(S, d, seed=1301 + n)
    ll_ref, g_ref = O.gp_loglik_grad_batch(X, Y[0], L, A, N, kid)
    ll, g = lib.loglik_grad_batch(X, Y[0], L, A, N, kid)
    assert relerr(ll, ll_ref) <= TOL_LL
    # same factorisation kernels as the value-only batch for n > 32; at n <= 32 that batch takes the warp-register path
    assert relerr(ll, lib.loglik_batch(X, Y[0], L, A, N, kid)) <= 1e-12
    scale = np.maximum(np.max(np.abs(g_ref), axis=1, keepdims=True), 1e-300)
    assert np.max(np.abs(g - g_ref) / scale) <= 1e-8, np.max(np.abs(g - g_ref) / scale)


def test_loglik_grad_discrete_and_per_sample_mean(lib):
    n, d, S = 90, 3, 5
    X, Y, _, _, _ = make_problem(n, d, seed=1401)
    X = X * 5.0
    mask = np.array([False, True, False])
    L, A, N = make_hyper_samples(S, d, seed=1402)
    Ymm = Y[0][None, :] - np.linspace(-0.5, 0.5, S)[:, None]
    ll_ref, g_ref = O.gp_loglik_grad_batch(X, Ymm, L * 3, A, N, 2, discrete_mask=mask)
    ll, g = lib.loglik_grad_batch(X, Ymm, L * 3, A, N, 2, discrete_mask=mask)
    assert relerr(ll, ll_ref) <= TOL_LL
    assert np.max(np.abs(g - g_ref) / np.max(np.abs(g_ref), axis=1, keepdims=True)) <= 1e-8


# ---------------------------------------------------------------------------------------------
# device-side candidate generation (SURVEY.md 8f rank 3): grid and uniform box
# ---------------------------------------------------------------------------------------------
def test_ei_score_grid_generated_on_device(lib):
    n, d = 150, 3
    X, Y, ls, amp, ns = make_problem(n, d, seed=1500)
    gp = lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], 2)
    lo, step, cnt = np.array([0.0, 0.125, -0.25]), np.array([0.0625, 0.125, 0.25]), np.array([17, 8, 7])
    # Iterators.product order: first dimension fastest (exact dyadic arithmetic -> host grid == device grid)
    idx = np.arange(int(np.prod(cnt)))
    pts = np.stack([lo[0] + step[0] * (idx % cnt[0]), lo[1] + step[1] * ((idx // cnt[0]) % cnt[1]),
                    lo[2] + step[2] * (idx // (cnt[0] * cnt[1]))])
    best = float(np.quantile(Y[0], 0.7))
    lb, ub = np.zeros(d), np.ones(d)                                   # third dimension partly out of bounds -> 0.
    ref, bv_ref, bi_ref = lib.ei_score([gp], 1, 1, pts, [1.0], best, None, lb, ub)
    acq, bv, bi, bx = lib.ei_score_grid([gp], 1, 1, lo, step, cnt, [1.0], best, None, lb, ub, want_acq=True)
    assert np.array_equal(acq, ref) and bi == bi_ref and bv == bv_ref and np.array_equal(bx, pts[:, bi])
    # shards of the index range reproduce the unsharded call (multi-GPU sharding by index block)
    cut = 431
    a0, v0, i0, _ = lib.ei_score_grid([gp], 1, 1, lo, step, cnt, [1.0], best, None, lb, ub, first=0, M=cut, want_acq=True)
    a1, v1, i1, x1 = lib.ei_score_grid([gp], 1, 1, lo, step, cnt, [1.0], best, None, lb, ub, first=cut, want_acq=True)
    assert np.array_equal(np.concatenate([a0, a1]), ref)
    assert (i0 if v0 >= v1 else i1) == bi_ref
    assert np.array_equal(x1, pts[:, i1])
    gp.free()


def test_ei_score_uniform_generated_on_device(lib):
    n, d, M = 200, 5, 20000
    X, Y, ls, amp, ns = make_problem(n, d, seed=1600)
    gp = lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], 0)
    lb, ub = np.full(d, 0.1), np.array([0.9, 1.0, 0.7, 0.95, 0.8])
    pts = lib.uniform_candidates(1234, 0, M, lb, ub)                    # host reproduction of the counter hash
    assert pts.min() >= 0.1 and np.all(pts.max(axis=1) <= ub)
    assert abs(pts.mean() - 0.5 * (lb + ub).mean()) < 0.01
    best = float(np.quantile(Y[0], 0.8))
    ref, bv_ref, bi_ref = lib.ei_score([gp], 1, 1, pts, [1.0], best, None, lb, ub)
    acq, bv, bi, bx = lib.ei_score_uniform([gp], 1, 1, 1234, M, lb, ub, [1.0], best, None, want_acq=True)
    assert np.array_equal(acq, ref) and bi == bi_ref and bv == bv_ref and np.array_equal(bx, pts[:, bi])
    a1, v1, i1, x1 = lib.ei_score_uniform([gp], 1, 1, 1234, 5000, lb, ub, [1.0], best, None, first=15000, want_acq=True)
    assert np.array_equal(a1, ref[15000:]) and i1 == 15000 + int(np.argmax(ref[15000:]))
    gp.free()


# ---------------------------------------------------------------------------------------------
# device-resident lock-step multi-start optimiser (SURVEY.md 8f rank 3)
# ---------------------------------------------------------------------------------------------
def test_multistart_on_device_matches_host_driver(lib):
    """Same algorithm as the host-side batched L-BFGS of the mirror (boss_b200.batched_lbfgs_maximize), which
    calls boss_ei_value_grad per evaluation: the device-resident driver must land on the same optima."""
    import boss_b200 as B
    n, d, M = 120, 3, 96
    X, Y, ls, amp, ns = make_problem(n, d, seed=1700)
    gp = lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], 2)
    post = O.posterior_fit(X, Y[0], ls[0], amp[0], ns[0], 2)
    best = float(np.quantile(Y[0], 0.7))
    lb, ub = np.zeros(d), np.ones(d)
    starts = B.generate_LHC((lb, ub), M, np.random.default_rng(1))
    Xd, fd, bx, bv, bi, evals = lib.ei_maximize_multistart([gp], 1, 1, starts, [1.0], best, None, lb, ub, iters=40)
    vg = lambda Z: lib.ei_value_grad([gp], 1, 1, Z, [1.0], best, None, lb, ub)
    Xh, fh = B.batched_lbfgs_maximize(vg, starts, lb, ub, iters=40)
    assert np.all(Xd >= lb[:, None]) and np.all(Xd <= ub[:, None])
    f0, _, _ = lib.ei_score([gp], 1, 1, starts, [1.0], best, None, lb, ub)
    assert np.all(fd >= f0 - 1e-15)                                   # monotone: never worse than the start
    assert np.max(fd) >= np.max(f0) and bi == int(np.argmax(fd)) and bv == fd[bi] and np.array_equal(bx, Xd[:, bi])
    assert abs(np.max(fd) - np.max(fh)) <= 1e-6 * np.max(fh)           # same best optimum as the host driver
    close = np.abs(fd - fh) <= 1e-6 * np.maximum(np.abs(fh), 1e-12)
    assert close.mean() >= 0.9                                        # start by start, up to line-search round-off
    ref, _, _ = O.ei_acquisition([[post]], Xd, [1.0], best, None, lb, ub)
    m = ref > 1e-30 * ref.max()
    assert relerr(fd[m], ref[m]) <= TOL_POST                           # reported values are the acquisition at x_out
    assert 3 <= evals < 41 * 12          # compaction: only starts still backtracking are re-evaluated
    # affine prior mean evaluated on the device == the same mean passed as host arrays to boss_ei_value_grad
    aff = np.array([[0.2, 0.5, -0.3, 0.1]])
    pm = lambda Z: (aff[0, 0] + aff[0, 1:] @ Z)[None, :]
    pmg = lambda Z: np.broadcast_to(aff[0, 1:][None, :, None], (1, d, Z.shape[1]))
    vg2 = lambda Z: lib.ei_value_grad([gp], 1, 1, Z, [1.0], best, None, lb, ub, prior_mean_s=pm(Z), prior_mean_grad_s=pmg(Z))
    Xa, fa, _, bva, _, _ = lib.ei_maximize_multistart([gp], 1, 1, starts, [1.0], best, None, lb, ub, iters=30,
                                                      prior_mean_affine=aff)
    Xh2, fh2 = B.batched_lbfgs_maximize(vg2, starts, lb, ub, iters=30)
    assert abs(bva - np.max(fh2)) <= 1e-6 * np.max(fh2)
    chk, _ = vg2(Xa)
    assert relerr(fa, chk) <= 1e-11      # device fma chain vs numpy for the affine mean: last-bit differences only
    gp.free()


def test_multistart_discrete_rounding_and_failure(lib):
    n, d = 60, 2
    X, Y, ls, amp, ns = make_problem(n, d, seed=1800)
    X = X * 6.0
    mask = np.array([True, False])
    gp = lib.gp_fit(X, Y[0], ls[0] * 4, amp[0], ns[0], 2, discrete_mask=mask)
    lb, ub = np.zeros(d), np.full(d, 6.0)
    starts = np.random.default_rng(3).random((d, 40)) * 6.0
    Xd, fd, bx, bv, bi, _ = lib.ei_maximize_multistart([gp], 1, 1, starts, [1.0], float(np.median(Y[0])), None, lb, ub,
                                                       iters=25, discrete_mask=mask)
    assert np.array_equal(Xd[0], np.round(Xd[0]))                      # rounded like optimization.jl:116
    chk, _, _ = lib.ei_score([gp], 1, 1, Xd, [1.0], float(np.median(Y[0])), None, lb, ub)
    assert np.array_equal(chk, fd)                                     # re-evaluated after rounding
    gp.free()


# ---------------------------------------------------------------------------------------------
# batched posterior fit (BI samples x slices)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,d,kid,S", [(20, 2, 0, 7), (200, 3, 2, 12), (520, 4, 1, 5)])
def test_fit_batch_matches_single_fits(lib, n, d, kid, S):
    X, Y, _, _, _ = make_problem(n, d, seed=2100 + n)
    L, A, N = make_hyper_samples(S, d, seed=2101 + n)
    Ymm = Y[0][None, :] - np.linspace(-0.3, 0.3, S)[:, None]
    gps = lib.gp_fit_batch(X, Ymm, L, A, N, kid)
    assert len(gps) == S and all(g is not None for g in gps)
    Xs = np.random.default_rng(5).random((d, 400))
    for s in (0, S // 2, S - 1):
        post = O.posterior_fit(X, Ymm[s], L[s], A[s], N[s], kid)
        mu, var, _ = lib.gp_predict(gps[s], Xs)
        mr, vr, _ = O.mean_and_var(post, Xs)
        assert relerr(mu, mr) <= TOL_POST and relerr(var, vr) <= TOL_POST
        ll = O.gp_loglik(X, Ymm[s], L[s], A[s], N[s], kid)
        assert abs(gps[s].loglik - ll) <= TOL_LL * abs(ll)
        assert lib.gp_append(gps[s], Xs[:, 0], 0.1)          # handles from the batch are full handles
    best = float(np.median(Y[0]))
    posts = [[O.posterior_fit(X, Ymm[s], L[s], A[s], N[s], kid)] for s in range(S)]
    gps2 = lib.gp_fit_batch(X, Ymm, L, A, N, kid)
    acq, _, bi = lib.ei_score(gps2, 1, S, Xs, [1.0], best, None)          # BI average over the S samples
    ref, _, _ = O.ei_acquisition(posts, Xs, [1.0], best, None)
    m = ref > 1e-200
    assert relerr(acq[m], ref[m]) <= TOL_POST and bi == O.julia_argmax_fast(ref)
    for g in gps + gps2:
        g.free()


def test_fit_batch_reports_non_pd_samples(lib):
    X = np.zeros((1, 40)); y = np.arange(40.0)
    gps = lib.gp_fit_batch(X, y, np.array([[1.0], [1.0]]), np.array([1e6, 1.0]), np.array([0.0, 0.5]), 0)
    assert gps[0] is None and gps[1] is not None
    gps[1].free()


# ---------------------------------------------------------------------------------------------
# adjudication: the restated reference path is itself only accurate to ~cond(K) eps.  Against an
# extended-precision evaluation (x87 long double, oracle.adjudicator_longdouble) the CUDA path must be at least
# as close to the exact value as the restated reference is (up to a small factor) -- evidence that the residual
# GPU-vs-oracle differences are rounding noise of either side, not a systematic deviation.
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,d,kid", [(400, 4, 2), (700, 6, 0), (1024, 8, 1)])
def test_cuda_as_close_to_extended_precision_truth_as_the_oracle(lib, n, d, kid):
    X, Y, ls, amp, ns = make_problem(n, d, seed=2500 + n)
    Xs = np.random.default_rng(9).random((d, 256))
    mu_t, var_t, ll_t = O.adjudicator_longdouble(X, Y[0], ls[0], amp[0], ns[0], kid, Xs)
    post = O.posterior_fit(X, Y[0], ls[0], amp[0], ns[0], kid)
    mu_o, var_o, _ = O.mean_and_var(post, Xs)
    ll_o = O.gp_loglik(X, Y[0], ls[0], amp[0], ns[0], kid)
    gp = lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], kid)
    mu_g, var_g, _ = lib.gp_predict(gp, Xs)
    ll_g = lib.loglik_batch(X, Y[0], ls[0][None, :], amp[:1], ns[:1], kid)[0]
    e = lambda a, t: float(np.max(np.abs(a - t) / np.abs(t)))
    assert e(mu_g, mu_t) <= max(4 * e(mu_o, mu_t), 1e-12), (e(mu_g, mu_t), e(mu_o, mu_t))
    assert e(var_g, var_t) <= max(4 * e(var_o, var_t), 1e-11), (e(var_g, var_t), e(var_o, var_t))
    assert abs(ll_g - ll_t) <= max(4 * abs(ll_o - ll_t), 1e-12 * abs(ll_t))
    assert abs(gp.loglik - ll_t) <= max(4 * abs(ll_o - ll_t), 1e-12 * abs(ll_t))
    assert e(mu_g, mu_t) <= 1e-9 and e(var_g, var_t) <= 1e-9 and abs(ll_g - ll_t) <= 1e-8 * abs(ll_t)
    gp.free()


def test_fast_kernel_fn(lib):
    """Device exp(-t) / sqrt / kappa used by the kernel-matrix stages (table + degree-6 polynomial; MUFU seed +
    Goldschmidt step) against numpy and 40-digit arithmetic."""
    import mpmath as mp
    mp.mp.dps = 40
    rng = np.random.default_rng(0)
    t = np.concatenate([[0.0, 1e-300, 1e-17, 1e-8, 0.5, 1.0, 699.999, 700.0, 700.5, 1e4],
                        rng.random(200000) * 60.0, 10.0 ** rng.uniform(-12, 2.8, 200000)])
    got = lib.dbg_kernel_fn(0, t)
    ref = np.exp(-t)
    live = t < 700.0
    rel = np.abs(got[live] - ref[live]) / ref[live]
    assert rel.max() <= 1e-15, rel.max()                 # vs numpy (itself ~0.5 ulp)
    idx = np.argsort(-rel)[:50]                          # worst cases against 40-digit arithmetic
    worst = max(abs(mp.mpf(float(got[live][i])) - mp.exp(-mp.mpf(float(t[live][i])))) / mp.exp(-mp.mpf(float(t[live][i]))) for i in idx)
    assert worst <= 6e-16, worst
    assert np.all(got[~live] == 0.0) and got[0] == 1.0

    x = np.concatenate([[1e-270, 1e-100, 0.25, 1.0, 2.0, 4.0, 1e100, 1e300], 10.0 ** rng.uniform(-30, 30, 200000),
                        rng.random(200000) * 100.0])
    s = lib.dbg_kernel_fn(1, x)
    rel = np.abs(s - np.sqrt(x)) / np.sqrt(x)            # numpy sqrt is correctly rounded
    assert rel.max() <= 2.3e-16, rel.max()               # <= 1 ulp
    assert np.allclose(lib.dbg_kernel_fn(1, np.array([0.0, 5e-324, 1e-300])), 1e-145, rtol=1e-9, atol=0)

    d2 = np.concatenate([[0.0, 1e-300, 1e-30, 1e-16], rng.random(100000) * 40.0, 10.0 ** rng.uniform(-20, 4, 100000)])
    r = np.sqrt(d2)
    want = {2: np.exp(-0.5 * d2), 3: (1 + np.sqrt(3) * r) * np.exp(-np.sqrt(3) * r),
            4: (1 + np.sqrt(5) * r + 5 * d2 / 3) * np.exp(-np.sqrt(5) * r),
            5: -np.exp(-0.5 * d2), 6: -3 * np.exp(-np.sqrt(3) * r),
            7: -(5 / 3) * (1 + np.sqrt(5) * r) * np.exp(-np.sqrt(5) * r)}
    for which, w in want.items():
        g = lib.dbg_kernel_fn(which, d2)
        ok = np.abs(w) > 1e-290
        assert np.all(np.abs(g[ok] - w[ok]) <= 2e-15 * np.abs(w[ok])), which
        assert np.all(np.abs(g[~ok]) <= 1e-280), which


@pytest.mark.parametrize("n,d,S,reps", [(700, 5, 37, 12), (512, 6, 96, 40), (1024, 8, 64, 40), (1300, 3, 9, 12)])
def test_loglik_is_repeatable_and_split_invariant(lib, n, d, S, reps):
    """The factorisation runs as concurrent stream groups with shared-memory reuse inside the fused panel kernel and
    look-ahead warps inside the diagonal-block kernel: a missing barrier shows up as run-to-run differences (it did:
    the diagonal-tile publication in potrf_tile_kernel raced with late readers in ~1 of 5 calls at n = 1024, S = 64
    until it got its own barrier).  Every repetition, and every split of the batch (sub-batches land in different
    stream groups), must agree bitwise."""
    X, Y, _, _, _ = make_problem(n, d, seed=n)
    L, A, N = make_hyper_samples(S, d, seed=S)
    first = lib.loglik_batch(X, Y[0], L, A, N, lib.KERNEL_MATERN52)
    assert relerr(first, O.gp_loglik_batch(X, Y[0], L, A, N, O.KERNEL_MATERN52)) <= 1e-8
    for _ in range(reps):
        again = lib.loglik_batch(X, Y[0], L, A, N, lib.KERNEL_MATERN52)
        assert np.array_equal(first, again)
    h = S // 3
    parts = [lib.loglik_batch(X, Y[0], L[a:b], A[a:b], N[a:b], lib.KERNEL_MATERN52) for a, b in ((0, h), (h, S - 1), (S - 1, S))]
    assert np.array_equal(first, np.concatenate(parts))
    ll_g, _ = lib.loglik_grad_batch(X, Y[0], L, A, N, lib.KERNEL_MATERN52)     # same factorisation, gradient mode
    assert np.array_equal(first, ll_g)


@pytest.mark.parametrize("n,d", [(640, 5), (1500, 8)])
def test_fit_score_gradient_paths_are_repeatable(lib, n, d):
    """Same idea for the other kernel families (right-looking fit + triangular inverse, scoring, x-gradient, hyper-
    parameter gradient, batched fit, covariance): repeated calls on identical inputs must agree bit for bit."""
    X, Y, ls, amp, ns = make_problem(n, d, seed=n + 1)
    Xs = np.random.default_rng(n).random((d, 5000))
    best = float(np.quantile(Y[0], 0.8))
    L, A, N = make_hyper_samples(6, d, seed=n + 2)
    ref = None
    for rep in range(8):
        gp = lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], lib.KERNEL_MATERN52)
        Lf, Wf, al = lib.dbg_factors(gp)
        acq, bv, bi = lib.ei_score([gp], 1, 1, Xs, [1.0], best, None)
        val, grad = lib.ei_value_grad([gp], 1, 1, Xs[:, :900], [1.0], best, None)
        mu, cov, _ = lib.gp_cov(gp, Xs[:, :300])
        ll, llg = lib.loglik_grad_batch(X, Y[0], L, A, N, lib.KERNEL_MATERN52)
        gps = lib.gp_fit_batch(X, Y[0], L, A, N, lib.KERNEL_MATERN52)
        mu_b = np.stack([lib.gp_predict(g, Xs[:, :200])[0] for g in gps])
        for g in gps:
            g.free()
        gp.free()
        out = (Lf, Wf, al, acq, np.array([bv, bi]), val, grad, mu, cov, ll, llg, mu_b)
        if ref is None:
            ref = out
        else:
            for k, (a, b) in enumerate(zip(ref, out)):
                assert np.array_equal(a, b), (rep, k)


@pytest.mark.parametrize("d", [5, 9, 11, 12, 13, 17, 32])
def test_every_x_dim_padding_class(lib, d):
    """x_dim is padded to 2/4/6/8/12/16/32 inside the kernels (template instantiations): one pass over predict, EI
    value + x-gradient, log-likelihood and its hyper-parameter gradient at dimensions that land in each class."""
    n, M, S, kid = 150, 300, 5, lib.KERNEL_MATERN52
    X, Y, ls, amp, ns = make_problem(n, d, seed=40 + d)
    ls = ls * np.sqrt(d / 3.0)                       # keep the kernel matrix well away from the identity
    Xs = np.random.default_rng(d).random((d, M))
    gp = lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], kid)
    post = O.posterior_fit(X, Y[0], ls[0], amp[0], ns[0], kid)
    mu, var, st = lib.gp_predict(gp, Xs)
    mu_r, var_r, _ = O.mean_and_var(post, Xs)
    assert relerr(mu, mu_r) <= TOL_POST and relerr(var, var_r) <= TOL_POST and not st.any()
    best = float(np.quantile(Y[0], 0.7))
    val, grad = lib.ei_value_grad([gp], 1, 1, Xs, [1.0], best, None)
    val_r, grad_r = O.ei_value_grad([post], Xs, [1.0], best, None)
    assert relerr(val, val_r) <= TOL_POST
    assert np.max(np.abs(grad - grad_r) / np.max(np.abs(grad_r), axis=1, keepdims=True)) <= 1e-8
    L, A, N = make_hyper_samples(S, d, seed=d)
    L = L * np.sqrt(d / 3.0)
    ll, g = lib.loglik_grad_batch(X, Y[0], L, A, N, kid)
    ll_r, g_r = O.gp_loglik_grad_batch(X, Y[0], L, A, N, kid)
    assert relerr(ll, ll_r) <= TOL_LL
    assert np.max(np.abs(g - g_r) / np.linalg.norm(g_r, axis=1, keepdims=True)) <= 1e-8
    assert np.array_equal(ll, lib.loglik_batch(X, Y[0], L, A, N, kid))
    gp.free()


def test_small_n_append_and_multistart_paths_are_repeatable(lib):
    """Warp-register log-likelihood (n <= 32), rank-1 append chain, device-generated candidates and the device
    multi-start driver: bitwise repeatable."""
    X, Y, ls, amp, ns = make_problem(30, 2, seed=77)
    L, A, N = make_hyper_samples(300, 2, seed=78)
    first = lib.loglik_batch(X, Y[0], L, A, N, lib.KERNEL_MATERN52)
    for _ in range(30):
        assert np.array_equal(first, lib.loglik_batch(X, Y[0], L, A, N, lib.KERNEL_MATERN52))
    n, d = 300, 3
    X, Y, ls, amp, ns = make_problem(n + 40, d, seed=79)
    best = float(np.quantile(Y[0][:n], 0.8))
    lb, ub = np.zeros(d), np.ones(d)
    starts = np.random.default_rng(80).random((d, 200))
    ref = None
    for rep in range(6):
        gp = lib.gp_fit(X[:, :n], Y[0][:n], ls[0], amp[0], ns[0], lib.KERNEL_MATERN52)
        for k in range(n, n + 40):
            assert lib.gp_append(gp, X[:, k], Y[0][k])
        Lf, Wf, al = lib.dbg_factors(gp)
        _, bv, bi, bx = lib.ei_score_uniform([gp], 1, 1, 1234, 20000, lb, ub, [1.0], best, None)
        Xo, fo, bxo, bvo, bio, ev = lib.ei_maximize_multistart([gp], 1, 1, starts, [1.0], best, None, lb, ub, iters=15)
        gp.free()
        out = (Lf, Wf, al, np.array([bv, bi]), bx, Xo, fo, bxo, np.array([bvo, bio, ev]))
        if ref is None:
            ref = out
        else:
            for k, (a, b) in enumerate(zip(ref, out)):
                assert np.array_equal(a, b), (rep, k)


def test_construct_ei_testset_of_the_reference(lib):
    """test/unit/test/acquisitions/expected_improvement.jl:43-110 ("construct_ei(fitness, posterior, constraints,
    eps_samples, best_yet)") on the device.  The reference uses ParametricPosterior(f = identity, noise_std = [1, 1]):
    mean(x) = x, std = 1.  Here two GP slices whose only training point is far away (posterior = prior, variance
    a^2 = 1) carry the identity as host-evaluated prior mean.  Single posterior and 4 identical posteriors (the BI
    average), LinFitness([1, 0]) through boss_ei_score and NonlinFitness(x -> x[1]) through the device MC-EI."""
    gps = [lib.gp_fit(np.array([[1000.0], [1000.0]]), np.array([0.0]), [1.0, 1.0], 1.0, 0.1, 0) for _ in range(2)]
    eps = np.array([[0.422498, -1.33921, 0.490985, -0.951167], [-0.289737, 0.162767, -0.499742, 0.892919]])
    coefs = np.array([1.0, 0.0])

    def make(nonlin, n_post, y_max, best):
        sl = gps * n_post

        def out(x):
            Xs = np.array(x, dtype=np.float64)[:, None]
            pm = Xs.copy()                                    # prior mean = identity: (y_dim, M)
            if nonlin:
                a, _, _ = lib.mcei_score(sl, 2, n_post, Xs, 1, eps, best, y_max, c=coefs, prior_mean_s=pm)
            else:
                a, _, _ = lib.ei_score(sl, 2, n_post, Xs, coefs, best, y_max, prior_mean_s=pm)
            return float(a[0])
        return out

    for nonlin in (False, True):
        for n_post in (1, 4):
            out = make(nonlin, n_post, None, None)
            assert out([1.0, 1.0]) == out([1.0, 1.0]) and out([1.0, 1.0]) == 0.0
            out = make(nonlin, n_post, np.array([np.inf, 10.0]), None)
            assert out([1.0, 1.0]) == out([1.0, 1.0]) and out([1.0, 1.0]) > 0.0
            assert out([5.0, 1.0]) == out([10.0, 1.0]) == out([15.0, 1.0])
            assert out([1.0, 5.0]) > out([1.0, 10.0]) > out([1.0, 15.0])
            assert abs(out([1.0, 20.0])) <= 1e-8
            out = make(nonlin, n_post, None, 10.0)
            assert out([11.0, 1.0]) == out([11.0, 1.0]) and out([11.0, 1.0]) > 0.0
            assert out([5.0, 1.0]) < out([10.0, 1.0]) < out([15.0, 1.0])
            assert abs(out([0.0, 1.0])) <= 1e-8
            assert out([1.0, 5.0]) == out([1.0, 10.0]) == out([1.0, 15.0])
            out = make(nonlin, n_post, np.array([np.inf, 10.0]), 10.0)
            assert out([11.0, 1.0]) == out([11.0, 1.0]) and out([11.0, 1.0]) > 0.0
            assert out([5.0, 1.0]) < out([10.0, 1.0]) < out([15.0, 1.0])
            assert out([11.0, 5.0]) > out([11.0, 10.0]) > out([11.0, 15.0])
            assert abs(out([1.0, 1.0])) <= 1e-8 and abs(out([11.0, 20.0])) <= 1e-8
    for g in gps:
        g.free()
