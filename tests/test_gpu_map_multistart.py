"""GPU tests of the device MAP fit of the hyper-parameters (boss_gp_map_multistart, DESIGN.md 2.15): the same
algorithm as its host twin (batched_lbfgs_maximize per slice on loglik_grad_batch + a numpy log-space prior), values
that are the values at the returned points, start / slice / device independence bit for bit, priors, failures,
argument errors, every kernel, full size, and the mirror's OptimizationMAP / SampleOptMAP(algorithm="device")."""
import math
import os
import subprocess
import sys

import numpy as np
import pytest

import boss_b200 as B
from tests import map_multistart_oracle as T
from tests.util_problems import make_problem

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module", autouse=True)
def _init(lib):
    return lib


def _lognormal_tables(y_dim, d):
    kind = np.full((y_dim, d + 2), 2, dtype=np.int32)
    par = np.zeros((y_dim, d + 2, 2))
    par[:, :d] = (0.0, 0.7)
    par[:, d] = (0.0, 0.5)
    par[:, d + 1] = (math.log(0.1), 0.5)
    return kind, par


def _starts(y_dim, M, d, seed):
    rng = np.random.default_rng(seed)
    st = np.empty((y_dim, M, d + 2))
    st[..., :d] = np.exp(rng.normal(0.0, 0.7, (y_dim, M, d)))
    st[..., d] = np.exp(rng.normal(0.0, 0.5, (y_dim, M)))
    st[..., d + 1] = np.exp(rng.normal(math.log(0.1), 0.5, (y_dim, M)))
    return st


def _mirror_prior(kind, par, raw):
    """the mirror's densities (boss.jl_b200/types.py) summed over one slice's entries"""
    mk = {0: lambda a, b: B.Dirac(a), 1: B.Normal, 2: B.LogNormal, 3: B.Uniform}
    return sum(mk[int(k)](*p).logpdf(x) for k, p, x in zip(kind, par, raw))


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint64)


def _rel(a, b):
    return abs(a - b) / max(abs(b), 1e-300)


@pytest.fixture(scope="module")
def parity(lib):
    n, d, y_dim, M = 120, 3, 2, 64
    X, Y, _, _, _ = make_problem(n, d, seed=5, y_dim=y_dim)
    kind, par = _lognormal_tables(y_dim, d)
    st = _starts(y_dim, M, d, seed=6)
    dev = lib.gp_map_multistart(X, Y, kind, par, st, lib.KERNEL_MATERN52, iters=40)
    host = T.host_twin(lib, X, Y, kind, par, st, lib.KERNEL_MATERN52, iters=40)
    f0 = T.start_values(lib, X, Y, kind, par, st, lib.KERNEL_MATERN52)
    return X, Y, kind, par, st, dev, host, f0


def test_same_algorithm_as_the_host_twin(parity):
    X, Y, kind, par, st, dev, host, f0 = parity
    po, fo, bp, bv, bi, ev = dev
    hp, hf = host
    assert ev >= 1
    for i in range(Y.shape[0]):
        assert _rel(bv[i], hf[i].max()) <= 1e-6, (bv[i], hf[i].max())
        agree = np.abs(fo[i] - hf[i]) <= 1e-6 * np.abs(hf[i])
        assert agree.mean() >= 0.9, agree.mean()
        assert np.all(fo[i] >= f0[i] - 1e-12 * np.abs(f0[i]))


def test_reported_value_is_the_value_at_the_point(lib, parity):
    X, Y, kind, par, st, dev, host, f0 = parity
    po, fo, bp, bv, bi, _ = dev
    d = X.shape[0]
    for i in range(Y.shape[0]):
        ll, _ = lib.loglik_grad_batch(X, Y[i], po[i, :, :d], po[i, :, d], po[i, :, d + 1], lib.KERNEL_MATERN52)
        ref = ll + np.array([_mirror_prior(kind[i], par[i], p) for p in po[i]])
        np.testing.assert_allclose(fo[i], ref, rtol=1e-12)
        b = int(np.argmax(fo[i]))                       # first maximal
        assert bi[i] == b and bv[i] == fo[i, b]
        assert np.array_equal(_bits(bp[i]), _bits(po[i, b]))


def test_independent_of_other_starts_slices_and_devices(lib):
    n, d, y_dim, M = 90, 2, 2, 24
    X, Y, _, _, _ = make_problem(n, d, seed=11, y_dim=y_dim)
    kind, par = _lognormal_tables(y_dim, d)
    st = _starts(y_dim, M, d, seed=12)
    po, fo, bp, bv, bi, _ = lib.gp_map_multistart(X, Y, kind, par, st, lib.KERNEL_MATERN32, iters=25)
    # the same starts split over two calls
    a = lib.gp_map_multistart(X, Y, kind, par, st[:, :10], lib.KERNEL_MATERN32, iters=25)
    b = lib.gp_map_multistart(X, Y, kind, par, st[:, 10:], lib.KERNEL_MATERN32, iters=25)
    assert np.array_equal(_bits(po), _bits(np.concatenate([a[0], b[0]], axis=1)))
    assert np.array_equal(_bits(fo), _bits(np.concatenate([a[1], b[1]], axis=1)))
    # a y_dim = 2 call equals two y_dim = 1 calls
    for i in range(y_dim):
        s = lib.gp_map_multistart(X, Y[i:i + 1], kind[i:i + 1], par[i:i + 1], st[i:i + 1], lib.KERNEL_MATERN32, iters=25)
        assert np.array_equal(_bits(po[i]), _bits(s[0][0])) and np.array_equal(_bits(fo[i]), _bits(s[1][0]))
        assert bi[i] == s[4][0] and np.array_equal(_bits(bp[i]), _bits(s[2][0]))


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
from tests import test_gpu_map_multistart as G
from tests.util_problems import make_problem
lib.init_multi(2)
X, Y, _, _, _ = make_problem(100, 3, seed=4, y_dim=3)
kind, par = G._lognormal_tables(3, 3)
st = G._starts(3, 21, 3, seed=5)
out = []
for pin in (-1, 0):
    lib.set_device(pin)
    out.append(lib.gp_map_multistart(X, Y, kind, par, st, lib.KERNEL_MATERN52, iters=20))
for a, b in zip(*out):
    assert np.array_equal(G._bits(np.asarray(a, dtype=np.float64)), G._bits(np.asarray(b, dtype=np.float64)))
print("multi ok")
'''


@pytest.mark.skipif(_n_gpus() < 2, reason="needs >= 2 GPUs")
def test_two_devices_match_one_bit_for_bit():
    """(slice, start) ranges dealt to two devices under boss_init_multi equal the single-device call.  Runs in its own
    process, so the rest of the suite keeps driving one device."""
    r = subprocess.run([sys.executable, "-c", _MULTI, ROOT], capture_output=True, text=True, cwd=ROOT)
    assert r.returncode == 0 and "multi ok" in r.stdout, r.stdout + r.stderr


def _twin_best(lib, X, Y, kind, par, st, kid, mask=None, iters=20):
    dev = lib.gp_map_multistart(X, Y, kind, par, st, kid, mask, iters=iters)
    _, hf = T.host_twin(lib, X, Y, kind, par, st, kid, mask, iters=iters)
    for i in range(Y.shape[0]):
        assert _rel(dev[3][i], hf[i].max()) <= 1e-6, (dev[3][i], hf[i].max())
    return dev


def test_dirac_pinned_entries_come_back_exactly(lib):
    n, d, M = 70, 3, 16
    X, Y, _, _, _ = make_problem(n, d, seed=21, y_dim=2)
    kind, par = _lognormal_tables(2, d)
    kind[0, 1] = 0; par[0, 1] = (0.55, 0.0)            # one pinned lengthscale
    kind[:, d + 1] = 0; par[0, d + 1, 0] = 0.0; par[1, d + 1, 0] = 0.05     # noise pinned, to 0 in slice 0
    st = _starts(2, M, d, seed=22)
    st[0, :, 1] = -1.0                                  # ignored for a pinned entry
    po, fo, bp, bv, bi, _ = _twin_best(lib, X, Y, kind, par, st, lib.KERNEL_SE)
    assert np.all(po[0, :, 1] == 0.55) and np.all(po[0, :, d + 1] == 0.0) and np.all(po[1, :, d + 1] == 0.05)
    assert bp[0, 1] == 0.55 and bp[0, d + 1] == 0.0 and bp[1, d + 1] == 0.05


def test_uniform_support_is_never_left(lib):
    n, d, M = 80, 2, 24
    X, Y, _, _, _ = make_problem(n, d, seed=31)
    kind, par = _lognormal_tables(1, d)
    kind[0, :d] = 3; par[0, :d] = (0.2, 0.6)            # a tight box around lengthscales that want to grow
    kind[0, d] = 3; par[0, d] = (0.5, 1.5)
    st = _starts(1, M, d, seed=32)
    st[0, :, :d] = np.random.default_rng(33).uniform(0.2, 0.6, (M, d))
    st[0, :, d] = np.random.default_rng(34).uniform(0.5, 1.5, M)
    po, fo, *_ = _twin_best(lib, X, Y, kind, par, st, lib.KERNEL_MATERN52, iters=30)
    assert np.all(np.isfinite(fo))
    assert np.all((po[0, :, :d] >= 0.2) & (po[0, :, :d] <= 0.6))
    assert np.all((po[0, :, d] >= 0.5) & (po[0, :, d] <= 1.5))


@pytest.mark.parametrize("k", [1, 2], ids=["normal", "lognormal"])
def test_normal_and_lognormal_priors(lib, k):
    n, d, M = 80, 2, 16
    X, Y, _, _, _ = make_problem(n, d, seed=41)
    kind, par = _lognormal_tables(1, d)
    kind[0, :] = k
    par[0, :d] = (0.8, 0.4) if k == 1 else (0.0, 0.7)
    par[0, d] = (1.0, 0.5) if k == 1 else (0.0, 0.5)
    par[0, d + 1] = (0.1, 0.05) if k == 1 else (math.log(0.1), 0.5)
    st = _starts(1, M, d, seed=42)
    po, fo, *_ = _twin_best(lib, X, Y, kind, par, st, lib.KERNEL_MATERN52)
    ll, _ = lib.loglik_grad_batch(X, Y[0], po[0, :, :d], po[0, :, d], po[0, :, d + 1], lib.KERNEL_MATERN52)
    ref = ll + np.array([_mirror_prior(kind[0], par[0], p) for p in po[0]])
    np.testing.assert_allclose(fo[0], ref, rtol=1e-12)


def test_failed_starts_are_not_chosen_and_a_failed_slice_is_reported(lib):
    n, d, M = 40, 2, 12
    X, Y, _, _, _ = make_problem(n, d, seed=51, y_dim=2)
    Y[1, 7] = np.nan                                    # slice 1: every start fails
    kind, par = _lognormal_tables(2, d)
    st = _starts(2, M, d, seed=52)
    bad = np.arange(M) % 3 == 0                         # K numerically rank one: amplitude and lengthscales e^30
    st[0, bad, :d + 1] = math.exp(30.0)
    f0 = T.start_values(lib, X, Y, kind, par, st, lib.KERNEL_SE)
    assert np.all(np.isneginf(f0[0, bad])) and np.all(np.isfinite(f0[0, ~bad]))       # the setup fails where meant to
    po, fo, bp, bv, bi, _ = lib.gp_map_multistart(X, Y, kind, par, st, lib.KERNEL_SE, iters=20)
    assert np.all(np.isneginf(fo[0, bad])) and np.all(np.isfinite(fo[0, ~bad]))
    assert bi[0] >= 0 and not bad[bi[0]] and bv[0] == fo[0].max()
    assert bi[1] == -1 and bv[1] == -math.inf and np.all(np.isneginf(fo[1]))


def test_argument_errors(lib):
    n, d, M = 30, 2, 4
    X, Y, _, _, _ = make_problem(n, d, seed=61)
    kind, par = _lognormal_tables(1, d)
    st = _starts(1, M, d, seed=62)
    k2 = kind.copy(); k2[0, 0] = 4
    with pytest.raises(lib.BossError, match=r"\(-1\)"):
        lib.gp_map_multistart(X, Y, k2, par, st)
    for v in (0.0, -1.0, np.nan, np.inf):
        s2 = st.copy(); s2[0, 1, 2] = v
        with pytest.raises(lib.BossError, match=r"\(-1\)"):
            lib.gp_map_multistart(X, Y, kind, par, s2)
    with pytest.raises(lib.BossError, match=r"\(-1\)"):
        lib.gp_map_multistart(X, Y, kind, par, st[:, :0])
    X33 = np.random.default_rng(63).random((33, n))
    k33, p33 = _lognormal_tables(1, 33)
    with pytest.raises(lib.BossError, match=r"\(-1\)"):
        lib.gp_map_multistart(X33, Y, k33, p33, _starts(1, M, 33, seed=64))
    with pytest.raises(lib.BossError, match=r"\(-1\)"):
        lib.gp_map_multistart(X, Y, kind, par, st, kernel_id=99)
    Y17 = np.zeros((17, n))
    with pytest.raises(lib.BossError, match=r"\(-1\)"):
        lib.gp_map_multistart(X, Y17, np.full((17, d + 2), 2), np.tile(par, (17, 1, 1)), np.tile(st, (17, 1, 1)))
    Yc, kc, pc, sc = (np.ascontiguousarray(a, dtype=t) for a, t in ((Y, np.float64), (kind, np.int32),
                                                                    (par, np.float64), (st, np.float64)))
    rc = lib.lib.boss_gp_map_multistart(None, d, n, 1, Yc.ctypes.data, 2, None, kc.ctypes.data, pc.ctypes.data,
                                        sc.ctypes.data, M, 10, 8, None, None, None, None, None, None)
    assert rc == -1


@pytest.mark.parametrize("kernel", ["se", "m32", "m52", "m12", "rq", "discrete"])
def test_every_kernel_against_the_host_twin(lib, kernel):
    n, d, M = 60, 2, 12
    X, Y, _, _, _ = make_problem(n, d, seed=71)
    kid = {"se": lib.KERNEL_SE, "m32": lib.KERNEL_MATERN32, "m52": lib.KERNEL_MATERN52, "m12": lib.KERNEL_MATERN12,
           "rq": lib.kernel_rational_quadratic(1.5), "discrete": lib.KERNEL_MATERN52}[kernel]
    mask = None
    if kernel == "discrete":
        X[0] = np.round(X[0] * 4)
        mask = np.array([1, 0], dtype=np.uint8)
    kind, par = _lognormal_tables(1, d)
    st = _starts(1, M, d, seed=72)
    _twin_best(lib, X, Y, kind, par, st, kid, mask, iters=15)


def test_full_size(lib):
    n, d, M = 2048, 8, 16
    X, Y, _, _, _ = make_problem(n, d, seed=81)
    kind, par = _lognormal_tables(1, d)
    st = _starts(1, M, d, seed=82)
    _twin_best(lib, X, Y, kind, par, st, lib.KERNEL_MATERN52, iters=10)


# ---- the mirror ---------------------------------------------------------------------------------------------------
def _problem(noise=0.1, seed=0, n=20, y_dim=1):
    rng = np.random.default_rng(seed)
    f = lambda x: np.array([np.sin(x[0]) + 0.5 * np.cos(2 * x[1]), np.cos(x[0] * x[1] / 5)][:y_dim])
    dom = B.Domain(([0.0, 0.0], [10.0, 10.0]))
    X = B.generate_LHC(dom.bounds, n, rng)
    Y = np.stack([f(X[:, j]) for j in range(n)], axis=1)
    model = B.GaussianProcess(
        kernel=B.SqExponentialKernel(),
        lengthscale_priors=[B.mvlognormal([0.5, 0.5], [0.5, 0.5])] * y_dim,
        amplitude_priors=[B.LogNormal(0.0, 0.5)] * y_dim,
        noise_std_priors=[B.Dirac(noise)] * y_dim)
    return B.BossProblem(f, dom, B.ExpectedImprovement(B.LinFitness([1.0] + [0.0] * (y_dim - 1))), model,
                         B.ExperimentData(X, Y))


@pytest.mark.parametrize("y_dim", [1, 2])
def test_mirror_optimization_map_and_sample_opt_map(y_dim):
    prob = _problem(seed=8, n=40, y_dim=y_dim)
    ll = B.model_loglike(prob.model, prob.data)
    host = B.estimate_parameters(B.OptimizationMAP(multistart=12, iters=30, seed=21, algorithm="lbfgs"), prob)
    dev = B.estimate_parameters(B.OptimizationMAP(multistart=12, iters=30, seed=21, algorithm="device"), prob)
    so_h = B.estimate_parameters(B.SampleOptMAP(samples=64, multistart=6, iters=30, seed=21), prob)
    so_d = B.estimate_parameters(B.SampleOptMAP(samples=64, multistart=6, iters=30, seed=21, algorithm="device"), prob)
    for r, ref in ((dev, host), (so_d, so_h)):
        assert abs(ll(r.params) - r.loglike) <= 1e-8 * abs(r.loglike)
        assert np.all(r.params.noise_std == 0.1)
        assert r.params.lengthscales.shape == (2, y_dim)
        assert r.loglike >= ref.loglike - 0.05 * abs(ref.loglike)
    allr = B.estimate_parameters(B.OptimizationMAP(multistart=5, iters=5, seed=3, algorithm="device"), prob,
                                 return_all=True)
    assert 1 <= len(allr) <= 5
    for r in allr:
        assert abs(ll(r.params) - r.loglike) <= 1e-8 * abs(r.loglike)


def _same(a, b):
    assert a.loglike == b.loglike
    for name in ("lengthscales", "amplitudes", "noise_std"):
        assert np.array_equal(getattr(a.params, name), getattr(b.params, name))


def test_mirror_falls_back_to_lbfgs_bit_for_bit():
    from boss_b200.types import Prior

    class HalfNormal(Prior):
        def rand(self, rng):
            return float(abs(rng.normal(0.0, 1.0)))

        def logpdf(self, x):
            return 0.5 * math.log(2 / math.pi) - 0.5 * x * x if x >= 0 else -math.inf

    prob = _problem(seed=9, n=30)
    prob.model.amplitude_priors = [HalfNormal()]
    a = B.estimate_parameters(B.OptimizationMAP(multistart=6, iters=10, seed=5, algorithm="lbfgs"), prob)
    b = B.estimate_parameters(B.OptimizationMAP(multistart=6, iters=10, seed=5, algorithm="device"), prob)
    _same(a, b)
    rng = np.random.default_rng(9)
    X = rng.random((2, 30)) * 4; Y = (2.0 * X[0] + np.sin(X[1]))[None, :]
    gp = B.GaussianProcess(kernel=B.Matern52Kernel(), lengthscale_priors=[B.mvlognormal([0, 0], [0.3, 0.3])],
                           amplitude_priors=[B.LogNormal()], noise_std_priors=[B.Dirac(0.1)])
    semi = B.Semiparametric(B.Parametric(lambda x, th: np.array([th[0] * x[0] + th[1]]),
                                         [B.Uniform(-3, 3), B.Uniform(-1, 1)],
                                         jacobian=lambda x, th: np.array([[x[0], 1.0]])), gp)
    sp = B.BossProblem(lambda x: x, B.Domain(([0.0, 0.0], [4.0, 4.0])), B.ExpectedImprovement(B.LinFitness([1.0])), semi,
                       B.ExperimentData(X, Y))
    a = B.estimate_parameters(B.SampleOptMAP(samples=32, multistart=4, iters=10, seed=5, algorithm="lbfgs"), sp)
    b = B.estimate_parameters(B.SampleOptMAP(samples=32, multistart=4, iters=10, seed=5, algorithm="device"), sp)
    _same(a, b)
    assert np.array_equal(a.params.theta, b.params.theta)


def test_bo_loop_with_the_device_fitter():
    prob = _problem(seed=8)
    n0 = len(prob.data)
    B.bo(prob, B.OptimizationMAP(multistart=8, iters=10, seed=0, algorithm="device"),
         B.OptimizationAM(multistart=32, iters=20, seed=0), B.IterLimit(2))
    assert len(prob.data) == n0 + 2 and prob.consistent
    assert np.isfinite(prob.params.loglike)
    assert abs(B.model_loglike(prob.model, prob.data)(prob.params.params) - prob.params.loglike) <= \
        1e-8 * abs(prob.params.loglike)
