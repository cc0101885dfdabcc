"""The log-likelihood gradient w.r.t. a parametric prior mean's theta (boss_gp_loglik_grad_batch_mean, DESIGN.md 2.13) and
the mirror's Semiparametric data_loglike_and_grad / gradient OptimizationMAP on it: against the numpy reference alpha^T J,
bit for bit against boss_gp_loglik_grad_batch and against itself over batches, strides, pointers and devices."""
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import boss_oracle as O
from tests import loglik_mean_grad_oracle as MG
from tests.test_loglik_mean_grad_host import _nonlinear_data, _nonlinear_model, linear_problem
from tests.util_problems import make_hyper_samples, make_problem

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def _case(n, d, S, k, seed, per_sample):
    """Training data, S hyper-parameter samples, per-sample delta = y - m(X; theta_s) and Jacobians J (k, n) / (S, k, n)."""
    X, Y, _, _, _ = make_problem(n, d, seed=seed)
    L, A, N = make_hyper_samples(S, d, seed=seed + 1)
    rng = np.random.default_rng(seed + 2)
    J = rng.standard_normal((S, k, n) if per_sample else (k, n))
    theta = rng.standard_normal((S, k)) * 0.3
    Jm = J if per_sample else np.broadcast_to(J, (S, k, n))
    Ymm = np.stack([Y[0] - theta[s] @ Jm[s] for s in range(S)])       # a mean linear in theta with Jacobian J_s
    return X, Ymm, J, L, A, N


def _raw(lib, X, Ymm, J, L, A, N, kid=2, mask=None, k=None, ldj=None, S=None, null=()):
    """The C call with every argument under the test's control -> (rc, loglik, grad, grad_mean)."""
    Xc = np.ascontiguousarray(X.T)
    n, d = Xc.shape
    S = L.shape[0] if S is None else S
    k = J.shape[-2] if k is None else k
    ldj = (0 if J.ndim == 2 else J.shape[-2] * n) if ldj is None else ldj
    Jc = np.ascontiguousarray(J)
    out, grad, gm = np.empty(max(S, 1)), np.empty((max(S, 1), d + 2)), np.empty((max(S, 1), max(k, 1)))
    p = lambda name, a: None if name in null or a is None else a.ctypes.data_as(lib._vp)
    dm = None if mask is None else np.ascontiguousarray(mask, dtype=np.uint8)
    Y = np.ascontiguousarray(Ymm)
    rc = lib.lib.boss_gp_loglik_grad_batch_mean(p("X", Xc), d, n, p("Y", Y), 0 if Y.ndim == 1 else n, p("J", Jc), k, ldj,
                                                p("L", L), p("A", A), p("N", N), kid, p("m", dm), S, p("ll", out),
                                                p("grad", grad), p("gm", gm))
    return rc, out, grad, gm


@pytest.mark.parametrize("kid", [O.KERNEL_SE, O.KERNEL_MATERN32, O.KERNEL_MATERN52])
@pytest.mark.parametrize("n", [20, 300, 1000])
def test_matches_the_reference_and_the_hyper_parameter_call(lib, kid, n):
    """grad_mean = alpha^T J to 1e-9 of its norm (k = 1, 2, 7; shared and per-sample J; a discrete dimension); loglik and
    grad equal boss_gp_loglik_grad_batch's bit for bit.  n = 1000, S = 9: 8 blocks, the 4-stream-group path."""
    d, S = 3, 9
    mask = np.array([0, 0, 1], dtype=np.uint8)
    for k in (1, 2, 7):
        for per_sample in (False, True):
            X, Ymm, J, L, A, N = _case(n, d, S, k, seed=10 * k + n, per_sample=per_sample)
            X[2] = np.round(X[2] * 3.0)
            ll, gr, gm = lib.loglik_grad_batch_mean(X, Ymm, J, L, A, N, kid, mask)
            ll0, gr0 = lib.loglik_grad_batch(X, Ymm, L, A, N, kid, mask)
            assert np.array_equal(_bits(ll), _bits(ll0)) and np.array_equal(_bits(gr), _bits(gr0))
            llr, gmr = MG.gp_loglik_mean_grad_batch(X, Ymm, J, L, A, N, kid, mask)
            assert np.all(np.isfinite(llr))
            err = np.max(np.abs(gm - gmr), axis=1) / np.maximum(np.linalg.norm(gmr, axis=1), 1e-300)
            assert np.max(err) <= 1e-9, (k, per_sample, err)


def test_batch_stride_and_pointer_independence(lib):
    """A sample's grad_mean is the same bits alone and inside a batch of 64; ldj = 0 equals the Jacobian repeated per
    sample (ldj = k*n) and a padded stride; the device-pointer variant equals the host one."""
    import torch
    n, d, S, k = 700, 4, 64, 5
    X, Ymm, J, L, A, N = _case(n, d, S, k, seed=3, per_sample=False)
    ll, gr, gm = lib.loglik_grad_batch_mean(X, Ymm, J, L, A, N, 2)
    for s in (0, 17, 63):
        a = lib.loglik_grad_batch_mean(X, Ymm[s:s + 1], J, L[s:s + 1], A[s:s + 1], N[s:s + 1], 2)
        assert np.array_equal(_bits(a[2][0]), _bits(gm[s])) and np.array_equal(_bits(a[1][0]), _bits(gr[s]))
    rep = np.ascontiguousarray(np.broadcast_to(J, (S, k, n)))
    _, _, gm_rep = lib.loglik_grad_batch_mean(X, Ymm, rep, L, A, N, 2)
    assert np.array_equal(_bits(gm_rep), _bits(gm))
    pad = np.zeros((S, k * n + 13)); pad[:, :k * n] = rep.reshape(S, k * n)
    rc, _, _, gm_pad = _raw(lib, X, Ymm, pad[:, None, :], L, A, N, k=k, ldj=k * n + 13)
    assert rc == 0 and np.array_equal(_bits(gm_pad), _bits(gm))
    # device pointers, per-sample J
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    tX, tY, tJ, tL, tA, tN = dev(X.T), dev(Ymm), dev(rep), dev(L), dev(A), dev(N)
    tll, tgr, tgm = (torch.empty(s, dtype=torch.float64, device="cuda") for s in ((S,), (S, d + 2), (S, k)))
    stream = torch.cuda.current_stream().cuda_stream
    lib.loglik_grad_batch_mean_dev(tX.data_ptr(), d, n, tY.data_ptr(), n, tJ.data_ptr(), k, k * n, tL.data_ptr(),
                                   tA.data_ptr(), tN.data_ptr(), 2, S, tll.data_ptr(), tgr.data_ptr(), tgm.data_ptr(),
                                   stream=stream)
    torch.cuda.synchronize()
    assert np.array_equal(_bits(tll.cpu().numpy()), _bits(ll)) and np.array_equal(_bits(tgr.cpu().numpy()), _bits(gr))
    assert np.array_equal(_bits(tgm.cpu().numpy()), _bits(gm))


def test_not_positive_definite_sample_and_argument_errors(lib):
    """A non-PD sample: -Inf, zero gradients, BOSS_NOT_POSDEF; the other samples are unaffected.  Argument errors;
    S = 0."""
    X = np.zeros((1, 150)); y = np.arange(150.0) / 150.0
    L, A, N = np.array([[1.0], [1.0], [0.7]]), np.array([1e6, 1.0, 2.0]), np.array([0.0, 0.5, 0.3])
    J = np.random.default_rng(0).standard_normal((3, 3, 150))
    rc, ll, gr, gm = _raw(lib, X, y, J, L, A, N, kid=0)
    assert rc == lib.BOSS_NOT_POSDEF
    assert ll[0] == -np.inf and np.all(gr[0] == 0.0) and np.all(gm[0] == 0.0)
    ok = lib.loglik_grad_batch_mean(X, y, J[1:], L[1:], A[1:], N[1:], 0)
    assert np.array_equal(_bits(ll[1:]), _bits(ok[0])) and np.array_equal(_bits(gm[1:]), _bits(ok[2]))
    X2, Ymm, J2, L2, A2, N2 = _case(40, 2, 3, 2, seed=5, per_sample=True)
    assert _raw(lib, X2, Ymm, J2, L2, A2, N2)[0] == 0
    for kw in (dict(k=0), dict(ldj=2 * 40 - 1), dict(ldj=-1), dict(null=("J",)), dict(null=("grad",)), dict(null=("gm",))):
        assert _raw(lib, X2, Ymm, J2, L2, A2, N2, **kw)[0] == -1, kw                 # BOSS_ERR_ARG
        assert "boss_gp_loglik_grad_batch_mean" in lib.last_error(), kw
    assert _raw(lib, X2, Ymm, J2, L2, A2, N2, S=0)[0] == 0


def test_mirror_data_loglike_and_grad_matches_central_differences(lib):
    """Semiparametric, y_dim = 2, a mean nonlinear in theta (theta[1] Dirac-pinned in the priors): the theta-gradient
    matches central differences of data_loglike in every entry, and the value equals data_loglike's."""
    import boss_b200 as B
    model, data = _nonlinear_model(B), _nonlinear_data(B)
    p = B.SemiparametricParams(np.array([1.2, 0.7, -0.4, 0.9]), np.array([[0.8, 1.1], [1.3, 0.6]]), np.array([1.0, 0.7]),
                               np.array([0.1, 0.1]))
    ll = B.data_loglike(model, data)
    v, g = B.data_loglike_and_grad(model, data)(p)
    assert abs(v - ll(p)) <= 1e-9 * abs(v)
    h = 1e-6
    for c in range(4):
        tp, tm = p.theta.copy(), p.theta.copy()
        tp[c] += h; tm[c] -= h
        fd = (ll(B.SemiparametricParams(tp, p.lengthscales, p.amplitudes, p.noise_std))
              - ll(B.SemiparametricParams(tm, p.lengthscales, p.amplitudes, p.noise_std))) / (2 * h)
        assert abs(g.theta[c] - fd) <= 1e-5 * max(1.0, abs(fd)), (c, g.theta[c], fd)


def test_gradient_optimization_map_of_semiparametric_models(lib):
    """Gradient OptimizationMAP reaches at least the compass search's log-likelihood (tolerance of
    test_gradient_optimization_map_and_sample_opt_map) on y = 2 x_1 + 0.5 + residual and on the reference's semiparametric
    testset problem, reports the value at its point, and SampleOptMAP reaches its best sample; without a Jacobian the
    "lbfgs" request is the compass search, bit for bit."""
    import boss_b200 as B
    prob = linear_problem(B)
    X = np.array([[2.0, 5.0, 8.0], [2.0, 5.0, 8.0]])
    fY = lambda x: np.array([np.sin(x[0]) + np.exp(x[1]), np.cos(x[0]) + np.exp(x[1])])
    predict = lambda x, th: np.array([th[0] * np.sin(x[0]) + th[1] * np.exp(x[1]), th[2] * np.cos(x[0]) + th[3] * np.exp(x[1])])
    jac = lambda x, th: np.array([[np.sin(x[0]), np.exp(x[1]), 0.0, 0.0], [0.0, 0.0, np.cos(x[0]), np.exp(x[1])]])
    ref_model = B.Semiparametric(B.Parametric(predict, [B.Normal()] * 4, jac),
                                 B.GaussianProcess(amplitude_priors=[B.LogNormal()] * 2,
                                                   lengthscale_priors=[B.mvlognormal([1.0, 1.0], [1.0, 1.0])] * 2,
                                                   noise_std_priors=[B.Dirac(1e-4)] * 2))
    ref_prob = B.BossProblem(lambda x: x, B.Domain(([0.0, 0.0], [10.0, 10.0])), B.ExpectedImprovement(B.LinFitness([1.0, 0.0])),
                             ref_model, B.ExperimentData(X, np.stack([fY(X[:, j]) for j in range(3)], axis=1)))
    for pb in (prob, ref_prob):
        ll = B.model_loglike(pb.model, pb.data)
        grad = B.estimate_parameters(B.OptimizationMAP(multistart=12, iters=30, seed=21, algorithm="lbfgs"), pb)
        comp = B.estimate_parameters(B.OptimizationMAP(multistart=12, iters=30, seed=21, algorithm="compass"), pb)
        samp = B.estimate_parameters(B.SamplingMAP(64, seed=21), pb)
        so = B.estimate_parameters(B.SampleOptMAP(samples=64, multistart=6, iters=30, seed=21), pb)
        for r in (grad, comp, so):
            assert abs(ll(r.params) - r.loglike) <= 1e-8 * abs(r.loglike)
        assert grad.loglike >= comp.loglike - 0.05 * abs(comp.loglike), (grad.loglike, comp.loglike)
        assert so.loglike >= samp.loglike - 1e-9
    nj = linear_problem(B, with_jacobian=False)
    a = B.estimate_parameters(B.OptimizationMAP(multistart=6, iters=20, seed=5, algorithm="lbfgs"), nj)
    b = B.estimate_parameters(B.OptimizationMAP(multistart=6, iters=20, seed=5, algorithm="compass"), nj)
    assert a.loglike == b.loglike and np.array_equal(a.params.theta, b.params.theta)
    assert np.array_equal(a.params.lengthscales, b.params.lengthscales) and np.array_equal(a.params.amplitudes, b.params.amplitudes)


def _n_gpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


_MULTI = r'''
import sys
import numpy as np
sys.path.insert(0, sys.argv[1])
import boss_b200
from boss_b200 import _lib as lib
from tests import test_gpu_loglik_mean_grad as T
lib.init_multi(2)
for per_sample in (False, True):
    X, Ymm, J, L, A, N = T._case(600, 3, 21, 4, seed=8, per_sample=per_sample)
    out = []
    for pin in (-1, 0):
        lib.set_device(pin)
        out.append(lib.loglik_grad_batch_mean(X, Ymm, J, L, A, N, 2))
    for a, b in zip(*out):
        assert np.array_equal(T._bits(a), T._bits(b))
print("multi ok")
'''


@pytest.mark.skipif(_n_gpus() < 2, reason="needs >= 2 GPUs")
def test_two_devices_match_one_bit_for_bit():
    """Sample ranges dealt to two devices under boss_init_multi (shared and per-sample J) equal the single-device call.
    Runs in its own process, so the rest of the suite keeps driving one device."""
    r = subprocess.run([sys.executable, "-c", _MULTI, ROOT], capture_output=True, text=True, cwd=ROOT)
    assert r.returncode == 0 and "multi ok" in r.stdout, r.stdout + r.stderr
