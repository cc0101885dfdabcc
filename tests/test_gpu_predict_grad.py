"""Posterior means, variances and their x-gradients (boss_gp_predict_grad, DESIGN.md 2.12) and the mirror's NonlinFitness
closures with `grad` differentiated through them: against the oracle's mean_var_grad and central differences, bit for
bit against boss_gp_predict, over chunks and devices, and OptimizationAM / SampleOptAM on a closure."""
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import boss_oracle as O
from tests import mcei_grad_oracle as MO
from tests.util_problems import make_problem, relerr

gpu = pytest.mark.gpu
TOL_POST = 1e-9
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _fit(lib, X, Y, ls, amp, ns, kid, S, mask=None):
    """S BI samples x y_dim slices, sample-major, on the device and in the oracle."""
    y_dim = Y.shape[0]
    gps, posts = [], []
    for s in range(S):
        lss = ls * (1 + 0.2 * s)
        gps += [lib.gp_fit(X, Y[i], lss[i], amp[i], ns[i], kid, discrete_mask=mask) for i in range(y_dim)]
        posts += [O.posterior_fit(X, Y[i], lss[i], amp[i], ns[i], kid, discrete_mask=mask) for i in range(y_dim)]
    assert all(g is not None for g in gps)
    return gps, posts


def _free(gps):
    for g in gps:
        g.free()


def _grad_err(g, ref):
    """max |g - ref| over each row's largest |ref| (rows: every leading index)"""
    scale = np.max(np.abs(ref), axis=-1, keepdims=True)
    scale = np.where(scale > 0, scale, 1.0)
    return float(np.max(np.abs(g - ref) / scale))


def _bits(v):
    return np.ascontiguousarray(v).view(np.int64 if np.asarray(v).dtype == np.float64 else np.int32)


@gpu
@pytest.mark.parametrize("kid", [0, 1, 2])
def test_matches_the_oracle(lib, kid):
    """y_dim = 3 x S = 2 posteriors, a discrete dimension, a prior mean and its gradient."""
    n, d, y_dim, S, M = 160, 4, 3, 2, 500
    X, Y, ls, amp, ns = make_problem(n, d, seed=500 + kid, y_dim=y_dim)
    X = X * 3.0
    mask = np.array([False, False, True, False])
    gps, posts = _fit(lib, X, Y, ls * 3.0, amp, ns, kid, S, mask)
    rng = np.random.default_rng(kid)
    Xs = rng.random((d, M)) * 3.0
    pm = rng.standard_normal((y_dim, M))
    pmg = rng.standard_normal((y_dim, d, M))
    mu, var, dmu, dvar, st = lib.gp_predict_grad(gps, y_dim, S, Xs, pm, pmg)
    assert mu.shape == (S * y_dim, M) and dmu.shape == (S * y_dim, d, M) and np.all(st == 0)
    for q in range(S * y_dim):
        i = q % y_dim
        mr, vr, dmr, dvr, sr = O.mean_var_grad(posts[q], Xs, pm[i], pmg[i])
        assert relerr(mu[q], mr) <= TOL_POST and relerr(var[q], vr) <= TOL_POST, q
        assert _grad_err(dmu[q], dmr) <= 1e-8 and _grad_err(dvar[q], dvr) <= 1e-8, q
        assert np.all(dvar[q, 2] == 0.0) and np.array_equal(dmu[q, 2], pmg[i, 2])    # discrete: the prior mean's only
    _free(gps)


@gpu
@pytest.mark.parametrize("kid", [0, 2])
def test_matches_central_differences_of_predict(lib, kid):
    n, d, M, h = 200, 3, 64, 1e-5
    X, Y, ls, amp, ns = make_problem(n, d, seed=600 + kid)
    gp = lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], kid)
    Xs = np.random.default_rng(9).random((d, M))
    _, _, dmu, dvar, _ = lib.gp_predict_grad([gp], 1, 1, Xs)
    for j in range(d):
        Xp = Xs.copy(); Xp[j] += h
        Xm = Xs.copy(); Xm[j] -= h
        mp, vp, _ = lib.gp_predict(gp, Xp)
        mm, vm, _ = lib.gp_predict(gp, Xm)
        for g, fd in ((dmu[0, j], (mp - mm) / (2 * h)), (dvar[0, j], (vp - vm) / (2 * h))):
            assert np.max(np.abs(g - fd)) <= 1e-6 * np.max(np.abs(fd)) + 1e-9, (j, np.max(np.abs(g - fd)))
    gp.free()


@gpu
def test_bits_equal_predict_with_clipping_and_failure(lib):
    """mu, var and status of every posterior are gp_predict's bit for bit.  Candidates on the training points of a
    nearly noiseless model get variances clipped to 0 (dvar == 0 there); a NaN coordinate fails (status 2, dvar 0)."""
    n, d, y_dim, S = 120, 2, 2, 2
    X, Y, ls, amp, ns = make_problem(n, d, seed=7, y_dim=y_dim, noise=1e-9)
    gps, _ = _fit(lib, X, Y, ls, amp, ns, 2, S)
    Xs = np.concatenate([X, np.random.default_rng(3).random((d, 100))], axis=1)
    Xs[1, n + 5] = np.nan
    M = Xs.shape[1]
    pm = np.random.default_rng(4).standard_normal((y_dim, M))
    mu, var, dmu, dvar, st = lib.gp_predict_grad(gps, y_dim, S, Xs, pm)
    clipped = 0
    for q in range(S * y_dim):
        m1, v1, s1 = lib.gp_predict(gps[q], Xs, pm[q % y_dim])
        assert np.array_equal(_bits(mu[q]), _bits(m1)) and np.array_equal(_bits(var[q]), _bits(v1))
        assert np.array_equal(st[q], s1)
        assert st[q, n + 5] == 2 and np.count_nonzero(st[q]) == 1 and np.all(dvar[q, :, n + 5] == 0.0)
        z = (var[q] == 0.0) & (st[q] == 0)      # var = a^2 - |W k*|^2 + 1e-18 is exactly 0 only when it was clipped
        assert np.all(dvar[q][:, z] == 0.0)
        clipped += int(z.sum())
    assert clipped > 0
    # a one-slice call over a prefix: the same numbers
    mu2, var2, dmu2, dvar2, _ = lib.gp_predict_grad(gps[:1], 1, 1, Xs[:, :3], pm[0, :3])
    assert np.array_equal(mu2[0], mu[0, :3]) and np.array_equal(dmu2[0], dmu[0, :, :3])
    _free(gps)


@gpu
@pytest.mark.parametrize("y_dim,S,d,M", [(2, 1, 3, 90_000), (8, 2, 32, 40_000)])
def test_chunks_from_pageable_and_pinned_memory_equal_small_calls(lib, y_dim, S, d, M):
    """Several chunks (the second shape, P = 16 and d = 32, runs at the capped chunk) from pageable and pinned memory
    equal the concatenation of calls of at most 20 000 candidates, bit for bit."""
    import torch
    X, Y, ls, amp, ns = make_problem(64, d, seed=8, y_dim=y_dim)
    gps, _ = _fit(lib, X, Y, ls, amp, ns, 2, S)
    Xs = np.random.default_rng(5).random((d, M))
    pm = np.random.default_rng(6).standard_normal((y_dim, M))
    full = lib.gp_predict_grad(gps, y_dim, S, Xs, pm)
    parts = [lib.gp_predict_grad(gps, y_dim, S, Xs[:, a:a + 20_000], pm[:, a:a + 20_000]) for a in range(0, M, 20_000)]
    pinned = torch.empty((M, d), dtype=torch.float64, pin_memory=True)
    pinned.copy_(torch.from_numpy(np.ascontiguousarray(Xs.T)))
    pin = lib.gp_predict_grad(gps, y_dim, S, pinned.numpy().T, pm)
    for k in range(5):
        cat = np.concatenate([p[k] for p in parts], axis=-1)
        assert np.array_equal(_bits(full[k]), _bits(cat)) and np.array_equal(_bits(pin[k]), _bits(cat)), k
    _free(gps)


@gpu
def test_argument_errors(lib):
    X, Y, ls, amp, ns = make_problem(40, 3, seed=9, y_dim=2)
    gps, _ = _fit(lib, X, Y, ls, amp, ns, 2, 1)
    Xs = np.random.default_rng(1).random((3, 20))
    Xc = np.ascontiguousarray(Xs.T)
    out = np.empty(20 * 2 * 3)
    raw = lambda arr, y_dim, S, M=20, dmu=out, dvar=None: lib.lib.boss_gp_predict_grad(
        arr, y_dim, S, lib._ptr(Xc), M, None, None, None, None, None if dmu is None else lib._ptr(dmu),
        None if dvar is None else lib._ptr(dvar), None)
    arr = lib._slice_array(gps)
    assert raw(arr, 2, 1, dmu=None) == -1 and "boss_gp_predict" in lib.last_error()     # neither gradient requested
    assert raw(None, 2, 1) == -1
    assert raw(arr, 0, 1) == -1 and raw(arr, 2, 0) == -1
    assert raw(arr, 2, 1, M=0) == 0                                                        # nothing to do
    nul = (lib._vp * 2)(gps[0].handle, None)
    assert raw(nul, 2, 1) == -1 and "NULL slice" in lib.last_error()
    with pytest.raises(lib.BossError, match="y_dim"):
        lib.gp_predict_grad((gps * 9)[:17], 17, 1, Xs)
    other = lib.gp_fit(np.random.default_rng(2).random((4, 30)), np.zeros(30), np.ones(4), 1.0, 0.1, 2)
    with pytest.raises(lib.BossError, match="x_dim"):
        lib.gp_predict_grad([gps[0], other], 2, 1, Xs)
    _free(gps + [other])   # x_dim <= 32 holds for every handle: boss_gp_fit refuses wider inputs


# ---- the mirror: NonlinFitness with grad ------------------------------------------------------------------------

EXPR = {1: dict(c0=1.0, c=[0.7, -0.2]),
        2: dict(c0=0.1, c=[1.0, 0.3], q=[0.0, -0.5], t=[0.0, 0.2]),
        3: dict(c0=0.0, c=[1.0, 0.8], t=[0.0, 0.1]),
        4: dict(c0=0.0, c=[1.0, 2.0], t=[0.0, 0.5])}
KIND = {1: "affine", 2: "quadratic", 3: "max", 4: "min"}


def _as_closure(B, expr):
    """The ExprFitness re-wrapped as an opaque NonlinFitness with the matching df/dy."""
    c0, c, q, t = expr.c0, expr.c, expr.q, expr.t
    return B.NonlinFitness(expr._eval, grad=lambda Z: MO._fit_and_grad(expr.kind_id, c0, c, q, t, Z)[1])


def _mirror_problem(B, kind, y_max=None, S=1):
    f = lambda x: np.array([np.sin(x[0]) + 0.1 * x[1], np.cos(x[0]) - 0.05 * x[1]])
    rng = np.random.default_rng(0)
    dom = B.Domain(([0.0, 0.0], [10.0, 10.0]))
    X = B.generate_LHC(dom.bounds, 20, rng)
    Y = np.stack([f(X[:, j]) for j in range(20)], axis=1)
    model = B.GaussianProcess(kernel=B.SqExponentialKernel(), lengthscale_priors=[B.mvlognormal([0.5, 0.5], [0.5, 0.5])] * 2,
                              amplitude_priors=[B.LogNormal(0.0, 0.5)] * 2, noise_std_priors=[B.Dirac(0.1)] * 2)
    e = EXPR[kind]
    prob = B.BossProblem(f, dom, B.ExpectedImprovement(B.ExprFitness(KIND[kind], e["c"], c0=e["c0"], q=e.get("q"),
                                                                     t=e.get("t")), eps_samples=100),
                         model, B.ExperimentData(X, Y), y_max=y_max)
    prob.params = B.estimate_parameters(B.SamplingMAP(64, seed=1), prob)
    if S > 1:
        q = prob.params.params
        plist = [B.GaussianProcessParams(q.lengthscales * (1.0 + 0.2 * s), q.amplitudes, q.noise_std) for s in range(S)]
        posts = B.model_posterior(prob.model, plist, prob.data)
    else:
        posts = B.model_posterior(prob)
    return prob, posts


@gpu
@pytest.mark.parametrize("kind", [1, 2, 3, 4])
@pytest.mark.parametrize("S", [1, 3])
def test_closure_matches_the_device_expression(lib, kind, S):
    """value_and_grad of the closure equals mcei_value_grad of the same expression to 1e-9 (away from kinks, where
    host and device may form y_k with and without an FMA), and its value equals acq(X) bit for bit."""
    import boss_b200 as B
    from boss_b200.acquisition import Acquisition
    prob, posts = _mirror_problem(B, kind, y_max=[np.inf, 0.6], S=S)
    ex = prob.acquisition.fitness
    eps = np.random.default_rng(3).standard_normal((2, 100 if S == 1 else S))
    best = B.best_so_far(prob, ex)
    acq_e = Acquisition(prob, posts, prob.acquisition, best, eps)
    acq_c = Acquisition(prob, posts, B.ExpectedImprovement(_as_closure(B, ex), eps_samples=100), best, eps)
    assert acq_e.expr is not None and acq_c.expr is None
    Xs = np.random.default_rng(4).random((2, 600)) * 11.0 - 0.5             # some out of bounds
    v_c, g_c = acq_c.value_and_grad(Xs)
    v_e, g_e = acq_e.value_and_grad(Xs)
    assert np.array_equal(_bits(v_c), _bits(acq_c(Xs)))
    p = prob.params.params
    post_o = [[O.posterior_fit(prob.data.X, prob.data.Y[i], p.lengthscales[:, i] * (1.0 + 0.2 * s), p.amplitudes[i],
                               p.noise_std[i], O.KERNEL_SE) for i in range(2)] for s in range(S)]
    keep = MO.kink_margin(post_o, Xs, kind, ex.c0, ex.c, ex.q, ex.t, eps, best) > 1e-6
    assert keep.sum() >= 400 and np.any(v_e[keep] > 0)
    assert np.all(np.abs(v_c - v_e)[keep] <= 1e-9 * np.maximum(np.abs(v_e[keep]), 1e-300))
    scale = np.maximum(np.max(np.abs(g_e[:, keep]), axis=1, keepdims=True), 1e-300)
    assert np.max(np.abs(g_c - g_e)[:, keep] / scale) <= 1e-9
    out = ~np.all((Xs >= 0.0) & (Xs <= 10.0), axis=0)
    assert out.any() and np.all(v_c[out] == 0.0) and np.all(g_c[:, out] == 0.0)


@gpu
def test_mirror_posterior_methods(lib):
    """mean_and_var_grad of a DefaultModelPosterior (one call for all slices) and of one slice: mean_and_var's numbers
    bit for bit, the gradients of gp_predict_grad, the vector forms equal to a column of the matrix forms."""
    import boss_b200 as B
    prob, post = _mirror_problem(B, 3)
    Xs = np.random.default_rng(6).random((2, 300)) * 10.0
    mu, var = post.mean_and_var(Xs)
    mu2, var2, dmu, dvar = post.mean_and_var_grad(Xs)
    assert np.array_equal(_bits(mu), _bits(mu2)) and np.array_equal(_bits(var), _bits(var2))
    ref = lib.gp_predict_grad([s.gp for s in post.slices], 2, 1, Xs)
    assert np.array_equal(dmu, ref[2]) and np.array_equal(dvar, ref[3]) and dmu.shape == (2, 2, 300)
    m1, v1, dm1, dv1 = post.slices[1].mean_and_var_grad(Xs)
    assert np.array_equal(m1, mu[1]) and np.array_equal(v1, var[1]) and np.array_equal(dm1, dmu[1])
    mv, vv, dmv, dvv = post.mean_and_var_grad(Xs[:, 7])
    assert np.array_equal(mv, mu[:, 7]) and np.array_equal(dmv, dmu[:, :, 7]) and dmv.shape == (2, 2)
    ms, vs, dms, dvs = post.slices[0].mean_and_var_grad(Xs[:, 7])
    assert ms == mu[0, 7] and vs == var[0, 7] and np.array_equal(dms, dmu[0, :, 7])
    bad = Xs[:, :4].copy()
    bad[0, 2] = np.nan
    with pytest.raises(ValueError, match="DomainError"):
        post.mean_and_var_grad(bad)
    with pytest.raises(ValueError, match="DomainError"):
        post.slices[0].mean_and_var_grad(bad)


@gpu
def test_closure_without_grad_still_raises(lib):
    import boss_b200 as B
    from boss_b200.acquisition import Acquisition
    prob, posts = _mirror_problem(B, 3)
    ex = prob.acquisition.fitness
    acq = Acquisition(prob, posts, B.ExpectedImprovement(B.NonlinFitness(ex._eval), eps_samples=100), 0.0)
    with pytest.raises(NotImplementedError):
        acq.value_and_grad(np.random.default_rng(1).random((2, 5)))


@gpu
@pytest.mark.parametrize("kind", [2, 3])
def test_optimization_am_and_sample_opt_am_on_a_closure(lib, kind):
    """OptimizationAM (host L-BFGS over value_and_grad) reaches at least the best start and the ExprFitness device
    driver's optimum; SampleOptAM runs on it too."""
    import boss_b200 as B
    from boss_b200 import acquisition_maximizers as AMs
    from boss_b200.acquisition import Acquisition
    prob, posts = _mirror_problem(B, kind)
    ex = prob.acquisition.fitness
    eps = np.random.default_rng(3).standard_normal((2, 100))
    best = B.best_so_far(prob, ex)
    acq_e = Acquisition(prob, posts, prob.acquisition, best, eps)
    acq_c = Acquisition(prob, posts, B.ExpectedImprovement(_as_closure(B, ex), eps_samples=100), best, eps)
    assert not acq_c.device_resident_ok()
    starts = B.generate_LHC(prob.domain.bounds, 32, np.random.default_rng(4))
    x_c, v_c = B.maximize_acquisition(AMs.OptimizationAM(starts, iters=40), prob, acq=acq_c)
    x_e, v_e = B.maximize_acquisition(AMs.OptimizationAM(starts, iters=40), prob, acq=acq_e)
    assert v_c >= np.max(acq_c(starts)) and v_c == acq_c(x_c)
    assert abs(v_c - v_e) <= 1e-6 * abs(v_e)
    x_s, v_s = B.maximize_acquisition(B.SampleOptAM(None, 2000, 16, iters=20, seed=5), prob, acq=acq_c)
    Xo, vals = B.maximize_acquisition(B.SamplingAM(None, 2000, seed=5), prob, return_all=True, acq=acq_c)
    assert v_s >= np.max(vals) and v_s == acq_c(x_s)


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
from tests import test_gpu_predict_grad as T
from tests.util_problems import make_problem
lib.init_multi(2)
X, Y, ls, amp, ns = make_problem(300, 4, seed=11, y_dim=3)
gps, _ = T._fit(lib, X, Y, ls, amp, ns, 2, 2)
Xs = np.random.default_rng(12).random((4, 50000))
pm = np.random.default_rng(13).standard_normal((3, 50000))
pmg = np.random.default_rng(14).standard_normal((3, 4, 50000))
out = []
for pin in (-1, 0):
    lib.set_device(pin)
    out.append(lib.gp_predict_grad(gps, 3, 2, Xs, pm, pmg))
for a, b in zip(*out):
    assert np.array_equal(T._bits(a), T._bits(b))
print("multi ok")
'''


@gpu
@pytest.mark.skipif(_n_gpus() < 2, reason="needs >= 2 GPUs")
def test_two_devices_match_one_bit_for_bit():
    """Split over two devices under boss_init_multi, the outputs equal the single-device call.  Runs in its own
    process, so the rest of the suite keeps driving one device."""
    r = subprocess.run([sys.executable, "-c", _MULTI, ROOT], capture_output=True, text=True, cwd=ROOT)
    assert r.returncode == 0 and "multi ok" in r.stdout, r.stdout + r.stderr
