"""x-gradient of the device Monte-Carlo EI (boss_mcei_value_grad, DESIGN.md 2.11) and the callers built on it:
boss_mcei_maximize_multistart, boss_mcei_score_topk and the mirror's OptimizationAM / SampleOptAM for an ExprFitness.
The numpy reference (tests/mcei_grad_oracle.py) is checked against central differences without a GPU; the GPU cases
check the device against the reference and against the value path bit for bit."""
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import boss_oracle as O
from tests import mcei_grad_oracle as MO
from tests.util_problems import make_problem

gpu = pytest.mark.gpu
TOL_POST = 1e-9
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# y_dim = 2 expressions of every kind (keyword arguments of the bindings)
EXPR = {1: dict(c0=1.0, c=[0.7, -0.2]),
        2: dict(c0=0.1, c=[1.0, 0.3], q=[0.0, -0.5], t=[0.0, 0.2]),
        3: dict(c0=0.0, c=[1.0, 0.8], t=[0.0, 0.1]),
        4: dict(c0=0.0, c=[1.0, 2.0], t=[0.0, 0.5])}


def _args(kind):
    e = EXPR[kind]
    return e["c0"], np.asarray(e["c"], float), np.asarray(e.get("q", [0.0, 0.0]), float), np.asarray(e.get("t", [0.0, 0.0]), float)


def _best(kind, Y, q=0.5):
    f = MO.fitness(kind, *_args(kind))
    return float(np.quantile([f(Y[:, j]) for j in range(Y.shape[1])], q))


# ---- the reference against central differences (no GPU) ---------------------------------------------------------

@pytest.mark.parametrize("kind", [1, 2, 3, 4])
@pytest.mark.parametrize("with_ymax", [False, True])
@pytest.mark.parametrize("S", [1, 3])
def test_reference_gradient_matches_central_differences(kind, with_ymax, S):
    """One posterior with K = 64 eps columns, or 3 BI posteriors with one column each; a linear prior mean on output 0
    with its gradient.  Candidates within 1e-4 of a kink (some |imp_k|, or a max / min gap) are skipped."""
    n, d, y_dim, M = 30, 3, 2, 16
    X, Y, ls, amp, ns = make_problem(n, d, seed=40 + kind, y_dim=y_dim)
    theta = np.array([0.3, -0.2, 0.1])
    Ymm = Y.copy()
    Ymm[0] -= theta @ X
    posts = [[O.posterior_fit(X, Ymm[i], ls[i] * (1 + 0.15 * s), amp[i], ns[i], O.KERNEL_MATERN52) for i in range(y_dim)]
             for s in range(S)]
    rng = np.random.default_rng(kind + 10 * S)
    eps = rng.standard_normal((y_dim, 64 if S == 1 else S))
    c0, c, q, t = _args(kind)
    f = MO.fitness(kind, c0, c, q, t)
    best = _best(kind, Y)
    y_max = [np.inf, float(np.quantile(Y[1], 0.6))] if with_ymax else None
    Xs = rng.random((d, M))
    pm = lambda Z: np.stack([theta @ Z, np.zeros(Z.shape[1])])
    pmg = np.zeros((y_dim, d, M))
    pmg[0] = theta[:, None]
    val, grad = MO.mc_ei_value_grad(posts, Xs, kind, c0, c, q, t, eps, best, y_max, pm(Xs), pmg)
    ref = O.mc_ei_acquisition(posts, Xs, f, eps, best, y_max, prior_mean_s=pm(Xs))
    assert np.allclose(val, ref, rtol=1e-9, atol=1e-15)
    keep = MO.kink_margin(posts, Xs, kind, c0, c, q, t, eps, best, pm(Xs)) > 1e-4
    assert keep.sum() >= M // 2
    assert np.any(grad[:, keep] != 0.0)
    h = 1e-6
    for j in range(d):
        Xp = Xs.copy(); Xp[j] += h
        Xm = Xs.copy(); Xm[j] -= h
        fp = O.mc_ei_acquisition(posts, Xp, f, eps, best, y_max, prior_mean_s=pm(Xp))
        fm = O.mc_ei_acquisition(posts, Xm, f, eps, best, y_max, prior_mean_s=pm(Xm))
        fd = (fp - fm) / (2 * h)
        assert np.allclose(grad[j, keep], fd[keep], rtol=2e-5, atol=1e-9), (j, grad[j, keep], fd[keep])


def test_reference_max_tie_takes_the_first_output():
    """At a tie of the max the reference (like the device) differentiates the first output's term."""
    Y = np.array([[1.0], [1.0]])[:, :, None]
    f, G = MO._fit_and_grad(3, 0.0, np.array([2.0, 3.0]), np.zeros(2), np.array([0.0, -1.0]), Y)
    assert f[0, 0] == 2.0 and G[0, 0, 0] == 2.0 and G[1, 0, 0] == 0.0


# ---- device --------------------------------------------------------------------------------------------------------

def _setup(lib, kid=2, S=1, n=150, d=3, M=400, seed=0, discrete_mask=None):
    y_dim = 2
    X, Y, ls, amp, ns = make_problem(n, d, seed=300 + seed, y_dim=y_dim)
    gps, posts = [], []
    for s in range(S):
        lss = ls * (1 + 0.2 * s)
        gps += [lib.gp_fit(X, Y[i], lss[i], amp[i], ns[i], kid, discrete_mask=discrete_mask) for i in range(y_dim)]
        posts.append([O.posterior_fit(X, Y[i], lss[i], amp[i], ns[i], kid, discrete_mask=discrete_mask)
                      for i in range(y_dim)])
    rng = np.random.default_rng(seed)
    eps = rng.standard_normal((y_dim, 200 if S == 1 else S))
    Xs = rng.random((d, M))
    return X, Y, gps, posts, eps, Xs


def _free(gps):
    for g in gps:
        g.free()


def _kw(kind):
    return dict(EXPR[kind])


def _grad_close(grad, gref, tol=1e-8):
    scale = np.max(np.abs(gref), axis=1, keepdims=True)
    scale = np.where(scale > 0, scale, 1.0)
    return float(np.max(np.abs(grad - gref) / scale))


@gpu
@pytest.mark.parametrize("kind", [1, 2, 3, 4])
@pytest.mark.parametrize("with_ymax", [False, True])
@pytest.mark.parametrize("S", [1, 3])
@pytest.mark.parametrize("kid", [0, 1, 2])
def test_value_grad_matches_reference(lib, kind, with_ymax, S, kid):
    """Four kinds x y_max x (K = 200 | 3 BI posteriors) x (SE, Matern 3/2, Matern 5/2), with a linear prior mean and
    its gradient on output 0.  The values are mcei_score's bit for bit."""
    d, M = 3, 400
    X, Y, gps, posts, eps, Xs = _setup(lib, kid, S, d=d, M=M, seed=kind + 4 * kid)
    theta = np.array([0.2, -0.3, 0.1])
    pm = np.stack([theta @ Xs, np.zeros(M)])
    pmg = np.zeros((2, d, M))
    pmg[0] = theta[:, None]
    best = _best(kind, Y, 0.7)
    y_max = [np.inf, float(np.quantile(Y[1], 0.6))] if with_ymax else None
    val, grad = lib.mcei_value_grad(gps, 2, S, Xs, kind, eps, best, y_max, prior_mean_s=pm, prior_mean_grad_s=pmg, **_kw(kind))
    c0, c, q, t = _args(kind)
    vref, gref = MO.mc_ei_value_grad(posts, Xs, kind, c0, c, q, t, eps, best, y_max, pm, pmg)
    assert np.any(vref > 0) and np.any(gref != 0)
    assert np.max(np.abs(val - vref)) <= TOL_POST * np.max(np.abs(vref))
    assert _grad_close(grad, gref) <= 1e-8
    acq, _, _ = lib.mcei_score(gps, 2, S, Xs, kind, eps, best, y_max, prior_mean_s=pm, **_kw(kind))
    assert np.array_equal(acq, val)
    _free(gps)


@gpu
def test_discrete_dimension_has_zero_derivative(lib):
    mask = np.array([True, False, False])
    X, Y, gps, posts, eps, Xs = _setup(lib, 2, 1, seed=21, discrete_mask=mask)
    best = _best(3, Y, 0.6)
    val, grad = lib.mcei_value_grad(gps, 2, 1, Xs, 3, eps, best, None, **_kw(3))
    vref, gref = MO.mc_ei_value_grad(posts, Xs, 3, *_args(3), eps, best, None)
    assert np.all(grad[0] == 0.0) and np.any(grad[1] != 0.0)
    assert np.max(np.abs(val - vref)) <= TOL_POST * np.max(np.abs(vref))
    assert _grad_close(grad[1:], gref[1:]) <= 1e-8
    _free(gps)


@gpu
@pytest.mark.parametrize("kind", [1, 2, 3, 4])
def test_pof_only_equals_the_closed_form_path(lib, kind):
    """best = None: PoF alone has no Monte-Carlo term; value and gradient are ei_value_grad's bit for bit."""
    X, Y, gps, posts, eps, Xs = _setup(lib, 2, 1, seed=31 + kind)
    y_max = [float(np.quantile(Y[0], 0.5)), float(np.quantile(Y[1], 0.6))]
    val, grad = lib.mcei_value_grad(gps, 2, 1, Xs, kind, eps, None, y_max, **_kw(kind))
    v2, g2 = lib.ei_value_grad(gps, 2, 1, Xs, [1.0, 0.0], None, y_max)
    assert np.array_equal(val, v2) and np.array_equal(grad, g2)
    _free(gps)


@gpu
def test_guards_give_a_zero_gradient(lib):
    """Out of bounds, cons_mask 0 and a failed variance (a NaN coordinate) give a zero gradient."""
    X, Y, gps, posts, eps, Xs = _setup(lib, 2, 1, M=8, seed=41)
    Xs = Xs.copy()
    Xs[0, 1] = 1.5            # out of the box
    Xs[1, 3] = np.nan         # fails _clip_var
    cm = np.ones(8, dtype=np.uint8)
    cm[5] = 0
    best = _best(3, Y, 0.0) - 1.0    # below every observation: every in-domain point has a positive EI and gradient
    val, grad = lib.mcei_value_grad(gps, 2, 1, Xs, 3, eps, best, None, lb=np.zeros(3), ub=np.ones(3), cons_mask=cm, **_kw(3))
    assert val[1] == 0.0 and val[5] == 0.0 and np.isneginf(val[3])
    assert np.all(grad[:, [1, 3, 5]] == 0.0)
    ok = [0, 2, 4, 6, 7]
    assert np.all(val[ok] > 0.0) and np.all(np.any(grad[:, ok] != 0.0, axis=0))
    _free(gps)


@gpu
@pytest.mark.parametrize("kind", [2, 3])
def test_gradient_does_not_depend_on_the_batch(lib, kind):
    """A point alone, in a 1 000-point batch and in a 40 000-point batch (quarter, narrow and wide shapes) gets the same
    gradient bit for bit."""
    n, d = 700, 4
    X, Y, gps, posts, eps, _ = _setup(lib, 2, 1, n=n, d=d, M=1, seed=51)
    big = np.random.default_rng(52).random((d, 40000))
    best = _best(kind, Y, 0.8)
    vb, gb = lib.mcei_value_grad(gps, 2, 1, big, kind, eps, best, None, **_kw(kind))
    for m in (1, 1000):
        v, g = lib.mcei_value_grad(gps, 2, 1, big[:, :m], kind, eps, best, None, **_kw(kind))
        assert np.array_equal(v, vb[:m]) and np.array_equal(g, gb[:, :m])
    assert np.any(gb[:, :1000] != 0)
    _free(gps)


@gpu
@pytest.mark.parametrize("S", [1, 3])
def test_multistart_matches_the_host_driver(lib, S):
    import boss_b200 as B
    n, d, M, kind = 120, 3, 96, 3
    X, Y, gps, posts, eps, _ = _setup(lib, 2, S, n=n, d=d, seed=61)
    best = _best(kind, Y, 0.7)
    lb, ub = np.zeros(d), np.ones(d)
    starts = B.generate_LHC((lb, ub), M, np.random.default_rng(1))
    kw = _kw(kind)
    Xd, fd, bx, bv, bi, evals = lib.mcei_maximize_multistart(gps, 2, S, starts, kind, eps, best, None, lb, ub, iters=40, **kw)
    vg = lambda Z: lib.mcei_value_grad(gps, 2, S, Z, kind, eps, best, None, lb=lb, ub=ub, **kw)
    Xh, fh = B.batched_lbfgs_maximize(vg, starts, lb, ub, iters=40)
    assert np.all(Xd >= lb[:, None]) and np.all(Xd <= ub[:, None])
    f0, _, _ = lib.mcei_score(gps, 2, S, starts, kind, eps, best, None, lb=lb, ub=ub, **kw)
    assert np.all(fd >= f0 - 1e-15)                                    # never worse than the start
    assert np.max(fd) > 0 and bi == int(np.argmax(fd)) and bv == fd[bi] and np.array_equal(bx, Xd[:, bi])
    assert abs(np.max(fd) - np.max(fh)) <= 1e-6 * np.max(fh)
    close = np.abs(fd - fh) <= 1e-6 * np.maximum(np.abs(fh), 1e-12)
    assert close.mean() >= 0.9
    chk, _, _ = lib.mcei_score(gps, 2, S, Xd, kind, eps, best, None, lb=lb, ub=ub, **kw)
    assert np.array_equal(chk, fd)                                     # f_out is the acquisition at x_out, bit for bit
    _free(gps)


@gpu
def test_multistart_discrete_rounding(lib):
    mask = np.array([True, False])
    X, Y, gps, posts, eps, _ = _setup(lib, 2, 1, n=60, d=2, seed=71, discrete_mask=mask)
    lb, ub = np.zeros(2), np.full(2, 6.0)
    starts = np.random.default_rng(3).random((2, 40)) * 6.0
    best = _best(2, Y, 0.5)
    Xd, fd, bx, bv, bi, _ = lib.mcei_maximize_multistart(gps, 2, 1, starts, 2, eps, best, None, lb, ub, iters=25,
                                                         discrete_mask=mask, **_kw(2))
    assert np.array_equal(Xd[0], np.round(Xd[0]))
    chk, _, _ = lib.mcei_score(gps, 2, 1, Xd, 2, eps, best, None, lb=lb, ub=ub, **_kw(2))
    assert np.array_equal(chk, fd)
    _free(gps)


def _ref_order(v):
    v = np.asarray(v, dtype=np.float64)
    nan = np.isnan(v)
    vv = np.where(nan, 0.0, v)
    return np.lexsort((np.arange(v.size), np.signbit(vv), -vv, ~nan))


def _bits(v):
    return np.ascontiguousarray(np.asarray(v, dtype=np.float64)).view(np.int64)


@gpu
def test_topk_is_the_head_of_the_host_order(lib):
    """200 000 candidates span several chunks; the k best pairs are the head of the host-ordered score vector."""
    M, kind = 200_000, 3
    X, Y, gps, posts, eps, _ = _setup(lib, 2, 1, n=1024, d=4, M=1, seed=81)
    Xs = np.random.default_rng(82).random((4, M))
    best = _best(kind, Y, 0.9)
    acq, _, _ = lib.mcei_score(gps, 2, 1, Xs, kind, eps, best, None, **_kw(kind))
    order = _ref_order(acq)
    for k in (1, 7, 1000, 8192):
        tv, ti = lib.mcei_score_topk(gps, 2, 1, Xs, kind, eps, best, None, k, **_kw(kind))
        assert np.array_equal(ti, order[:k]) and np.array_equal(_bits(tv), _bits(acq[order[:k]])), k
    for k in (0, 8193):
        with pytest.raises(lib.BossError):
            lib.mcei_score_topk(gps, 2, 1, Xs, kind, eps, best, None, k, **_kw(kind))
    with pytest.raises(lib.BossError):
        lib.mcei_score_topk(gps, 2, 1, Xs[:, :10], kind, eps, best, None, 11, **_kw(kind))
    _free(gps)


@gpu
def test_argument_errors(lib):
    X, Y, gps, posts, eps, Xs = _setup(lib, 2, 1, M=50, seed=91)
    lb, ub = np.zeros(3), np.ones(3)
    best = 0.0
    big = np.zeros((2, 4097))
    c = [1.0, 1.0]
    calls = [   # (kind, eps, S): bad kind (twice), more than 4096 eps columns, 200 eps columns for 3 BI posteriors
        lambda k, e, S: lib.mcei_value_grad(gps * S, 2, S, Xs, k, e, best, None, c=c),
        lambda k, e, S: lib.mcei_maximize_multistart(gps * S, 2, S, Xs, k, e, best, None, lb, ub, iters=2, c=c),
        lambda k, e, S: lib.mcei_score_topk(gps * S, 2, S, Xs, k, e, best, None, 3, c=c),
    ]
    for call in calls:
        for k, e, S in ((0, eps, 1), (5, eps, 1), (1, big, 1), (1, eps, 3)):
            with pytest.raises(lib.BossError, match=r"\(-1\)"):
                call(k, e, S)
    # NULL grad through the raw entry point
    arr = lib._slice_array(gps)
    Xc = np.ascontiguousarray(Xs.T)
    ep = np.ascontiguousarray(eps.T)
    b = np.array([best])
    rc = lib.lib.boss_mcei_value_grad(arr, 2, 1, lib._ptr(Xc), 50, None, None, 1, 0.0, None, None, None, lib._ptr(ep), 200,
                                      lib._ptr(b), None, None, None, None, None, None)
    assert rc == -1 and "grad is NULL" in lib.last_error()
    _free(gps)


def _mirror_problem():
    import boss_b200 as B
    f = lambda x: np.array([np.sin(x[0]) + 0.1 * x[1], np.cos(x[0]) - 0.05 * x[1]])
    rng = np.random.default_rng(0)
    dom = B.Domain(([0.0, 0.0], [10.0, 10.0]))
    X = B.generate_LHC(dom.bounds, 20, rng)
    Y = np.stack([f(X[:, j]) for j in range(20)], axis=1)
    model = B.GaussianProcess(kernel=B.SqExponentialKernel(), lengthscale_priors=[B.mvlognormal([0.5, 0.5], [0.5, 0.5])] * 2,
                              amplitude_priors=[B.LogNormal(0.0, 0.5)] * 2, noise_std_priors=[B.Dirac(0.1)] * 2)
    prob = B.BossProblem(f, dom, B.ExpectedImprovement(B.ExprFitness("max", [1.0, 0.8], t=[0.0, 0.1]), eps_samples=100),
                         model, B.ExperimentData(X, Y))
    prob.params = B.estimate_parameters(B.SamplingMAP(64, seed=1), prob)
    return prob


@gpu
def test_mirror_optimization_am_and_sample_opt_am_with_an_expr_fitness(lib):
    import boss_b200 as B
    from boss_b200 import acquisition_maximizers as AMs
    prob = _mirror_problem()
    acq = B.construct_acquisition(prob, eps=np.random.default_rng(3).standard_normal((2, 100)))
    assert acq.expr is not None and acq.device_resident_ok()
    am = AMs.OptimizationAM(32, iters=30, seed=4)
    starts = B.generate_LHC(prob.domain.bounds, 32, np.random.default_rng(4))
    x, v = B.maximize_acquisition(am, prob, acq=acq)
    assert v >= np.max(acq(starts)) and v == acq(x)
    val, grad = acq.value_and_grad(starts)
    assert np.array_equal(val, acq(starts)) and grad.shape == starts.shape
    # SampleOptAM: the starts are the head of a host sort of acq(X)
    sam = B.SampleOptAM(None, 3000, 16, iters=20, seed=5)
    x_new, v_new = B.maximize_acquisition(sam, prob, acq=acq)
    old = B.SampleOptAM(None, 3000, 16, iters=20, seed=5)
    Xo, vals = B.maximize_acquisition(old.sampler, prob, return_all=True, acq=acq)
    top_old = _ref_order(vals)[:16]
    top_new, tv = acq.topk(Xo, 16)
    assert np.array_equal(top_new, top_old) and np.array_equal(_bits(tv), _bits(vals[top_old]))
    x_old, v_old = B.maximize_acquisition(AMs.OptimizationAM(Xo[:, top_old], old.iters), prob, acq=acq)
    assert np.array_equal(x_new, x_old) and v_new == v_old and v_new >= vals[top_old[0]]


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
from tests import test_gpu_mcei_grad as T
lib.init_multi(2)
X, Y, gps, posts, eps, _ = T._setup(lib, 2, 1, n=300, d=3, M=1, seed=101)
Xs = np.random.default_rng(102).random((3, 50000))
best = T._best(3, Y, 0.8)
kw = T._kw(3)
starts = np.random.default_rng(103).random((3, 600))
lb, ub = np.zeros(3), np.ones(3)
out = []
for pin in (-1, 0):
    lib.set_device(pin)
    v, g = lib.mcei_value_grad(gps, 2, 1, Xs, 3, eps, best, None, **kw)
    tv, ti = lib.mcei_score_topk(gps, 2, 1, Xs, 3, eps, best, None, 1000, **kw)
    ms = lib.mcei_maximize_multistart(gps, 2, 1, starts, 3, eps, best, None, lb, ub, iters=20, **kw)
    out.append((v, g, tv, ti, ms[0], ms[1], ms[3], ms[4]))
for a, b in zip(*out):
    assert np.array_equal(np.asarray(a), np.asarray(b))
print("multi ok")
'''


@gpu
@pytest.mark.skipif(_n_gpus() < 2, reason="needs >= 2 GPUs")
def test_two_devices_match_one_bit_for_bit():
    """Value + gradient, top-k and the multi-start solve split over two devices equal the single-device call.  Runs in
    its own process, so the rest of the suite keeps driving one device."""
    r = subprocess.run([sys.executable, "-c", _MULTI, ROOT], capture_output=True, text=True, cwd=ROOT)
    assert r.returncode == 0 and "multi ok" in r.stdout, r.stdout + r.stderr
