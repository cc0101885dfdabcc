"""ExponentialKernel (Matern12, kernel_id 3) and RationalQuadraticKernel (registered ids) on the device: covariance
functions, fit and predict, the log-likelihood on every factorisation path and its gradients, the x-gradients, EI
scoring with screening, top-k, device candidates, the multi-start drivers, append, cov, the kernel-id rules, guard
bands, multi-device replication and the host mirror.  References: tests/kernels_more_oracle.py."""
import os
import subprocess
import sys

import numpy as np
import pytest

from tests import mcei_grad_oracle as MO
from tests.kernels_more_oracle import KERNEL_MATERN12, KERNELS, RQ, O, adjudicator_mean_var_loglik, kappa, \
    kappa_dr_over_r, kernel_name
from tests.util_problems import make_hyper_samples, make_problem

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
IDS = [kernel_name(k) for k in KERNELS]
TOL_POST, TOL_LL = 1e-9, 1e-8


def kid_of(lib, kernel):
    return lib.kernel_rational_quadratic(kernel.a) if isinstance(kernel, RQ) else kernel


def _close(a, ref, tol, scale=None):
    a, ref = np.asarray(a, float), np.asarray(ref, float)
    s = np.max(np.abs(ref)) if scale is None else scale
    return float(np.max(np.abs(a - ref))) <= tol * max(s, 1e-300)


def _fit(lib, kernel, n, d, seed, mask=None, noise=0.1):
    X, Y, ls, amp, ns = make_problem(n, d, seed=seed, noise=noise)
    gp = lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], kid_of(lib, kernel), mask)
    post = O.posterior_fit(X, Y[0], ls[0], amp[0], ns[0], kernel, mask)
    return X, Y, ls, amp, ns, gp, post


# ---- covariance functions ----------------------------------------------------------------------------------------

@pytest.mark.parametrize("kernel", KERNELS, ids=IDS)
def test_kernel_functions(lib, kernel):
    d2 = np.concatenate([[0.0, 1e-300, 1e-20, 1e-8], np.linspace(1e-3, 50.0, 2000), [300.0, 800.0]])
    kid = kid_of(lib, kernel)
    kr, dr = kappa(d2, kernel), kappa_dr_over_r(d2, kernel)
    tol = 2e-15 * (1.0 + np.sqrt(d2) + (d2 if isinstance(kernel, RQ) else 0.0))
    for which, ref in ((0, kr), (1, dr), (2, kr), (3, dr)):
        v = lib.dbg_kernel_fn_id(kid, which, d2)
        assert np.all(np.isfinite(v))
        ok = np.abs(v - ref) <= tol * np.abs(ref) + 1e-300
        assert ok.all(), (which, d2[~ok][:4], v[~ok][:4], ref[~ok][:4])
        if which in (0, 2):
            assert v[0] == 1.0
        else:
            assert v[0] == (0.0 if kernel == KERNEL_MATERN12 else -1.0)


def test_existing_ids_through_the_new_hook(lib):
    d2 = np.linspace(0.0, 20.0, 101)
    for kid in (0, 1, 2):
        assert np.array_equal(lib.dbg_kernel_fn_id(kid, 0, d2), lib.dbg_kernel_fn(2 + kid, d2))
        assert np.array_equal(lib.dbg_kernel_fn_id(kid, 1, d2), lib.dbg_kernel_fn(5 + kid, d2))


# ---- fit and predict ---------------------------------------------------------------------------------------------

SHAPES = [(1, 20), (3, 127), (5, 129), (8, 1000), (10, 20), (13, 127), (20, 129)]   # every DP in {2,...,32}


@pytest.mark.parametrize("kernel", KERNELS, ids=IDS)
@pytest.mark.parametrize("d,n", SHAPES)
def test_fit_predict_matches_oracle(lib, kernel, d, n):
    X, Y, ls, amp, ns, gp, post = _fit(lib, kernel, n, d, seed=d * 31 + n)
    Xs = np.random.default_rng(d + n).random((d, 300))
    Xs[:, :3] = X[:, :3]                        # candidates on training points
    mu, var, st = lib.gp_predict(gp, Xs)
    mu_r, var_r, st_r = O.mean_and_var(post, Xs)
    assert (st == 0).all() and (st_r == 0).all()
    assert _close(mu, mu_r, TOL_POST)
    assert _close(var, var_r, TOL_POST, scale=amp[0] ** 2)
    assert gp.loglik == pytest.approx(O.gp_loglik(X, Y[0], ls[0], amp[0], ns[0], kernel), rel=TOL_LL)
    if n <= 40:
        mu_a, var_a, ll_a = adjudicator_mean_var_loglik(X, Y[0], ls[0], amp[0], ns[0], kernel, Xs[:, :6], dps=40)
        assert _close(mu[:6], mu_a, TOL_POST) and _close(var[:6], var_a, TOL_POST, scale=amp[0] ** 2)
        assert gp.loglik == pytest.approx(ll_a, rel=TOL_LL)
    gp.free()


@pytest.mark.parametrize("kernel", KERNELS, ids=IDS)
def test_discrete_kernel_mask(lib, kernel):
    mask = np.array([True, False, True, False])
    X, Y, ls, amp, ns = make_problem(150, 4, seed=3)
    X[mask] = np.round(X[mask] * 4)
    gp = lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], kid_of(lib, kernel), mask)
    post = O.posterior_fit(X, Y[0], ls[0], amp[0], ns[0], kernel, mask)
    Xs = np.random.default_rng(4).random((4, 200)) * 4
    mu, var, _ = lib.gp_predict(gp, Xs)
    mu_r, var_r, _ = O.mean_and_var(post, Xs)
    assert _close(mu, mu_r, TOL_POST) and _close(var, var_r, TOL_POST, scale=amp[0] ** 2)
    gp.free()


# ---- log-likelihood on every factorisation path ------------------------------------------------------------------

def _ll_problem(n, d, S, seed):
    X, Y, _, _, _ = make_problem(n, d, seed=seed)
    L, A, N = make_hyper_samples(S, d, seed=seed + 1)
    return X, Y[0], L, A, N


@pytest.mark.parametrize("kernel", KERNELS, ids=IDS)
# n = 700 pads to 6 blocks, which still take the fused diagonal step (potrf_fused_kernel); n = 900 (8 blocks) runs the
# separate SYRK -> potrf_tile_kernel -> chol_panel_kernel chain
@pytest.mark.parametrize("n,path", [(20, "warp"), (300, "fused"), (700, "fused"), (900, "blocked")])
def test_loglik_paths(lib, kernel, n, path):
    X, y, L, A, N = _ll_problem(n, 5, 12, seed=n)
    ll = lib.loglik_batch(X, y, L, A, N, kid_of(lib, kernel))
    ref = O.gp_loglik_batch(X, y, L, A, N, kernel)
    assert np.all(np.isfinite(ref))
    assert np.max(np.abs(ll - ref) / np.abs(ref)) <= TOL_LL


@pytest.mark.parametrize("kernel", KERNELS, ids=IDS)
def test_fit_batch_bitwise_and_loglik(lib, kernel):
    X, y, L, A, N = _ll_problem(200, 4, 6, seed=9)
    kid = kid_of(lib, kernel)
    gps = lib.gp_fit_batch(X, y, L, A, N, kid)
    ll = lib.loglik_batch(X, y, L, A, N, kid)
    Xs = np.random.default_rng(10).random((4, 500))
    for s, g in enumerate(gps):
        one = lib.gp_fit_batch(X, y, L[s:s + 1], A[s:s + 1], N[s:s + 1], kid)[0]   # the same fit, one at a time
        assert g.loglik == ll[s] == one.loglik
        a, b = lib.gp_predict(g, Xs), lib.gp_predict(one, Xs)
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
        single = lib.gp_fit(X, y, L[s], A[s], N[s], kid)
        assert single.loglik == pytest.approx(ll[s], rel=1e-12)
        for h in (one, g, single):
            h.free()


# ---- hyper-parameter gradients -----------------------------------------------------------------------------------

@pytest.mark.parametrize("kernel", KERNELS, ids=IDS)
@pytest.mark.parametrize("n", [20, 300])
def test_loglik_grad(lib, kernel, n):
    X, y, L, A, N = _ll_problem(n, 3, 8, seed=n + 5)
    if kernel == KERNEL_MATERN12:
        X[:, 1] = X[:, 0]                          # a duplicated training point: g dq^2 -> 0
    ll, gr = lib.loglik_grad_batch(X, y, L, A, N, kid_of(lib, kernel))
    rl, rg = O.gp_loglik_grad_batch(X, y, L, A, N, kernel)
    assert np.all(np.isfinite(gr))
    assert np.max(np.abs(ll - rl) / np.abs(rl)) <= TOL_LL
    for s in range(len(ll)):
        assert np.max(np.abs(gr[s] - rg[s])) <= TOL_LL * np.linalg.norm(rg[s])


@pytest.mark.parametrize("kernel", KERNELS, ids=IDS)
def test_semiparametric_mean_grad(lib, kernel):
    X, y, L, A, N = _ll_problem(150, 3, 4, seed=21)
    J = np.stack([np.ones(150), X[0], X[1] ** 2])      # (k, n): row c is column c of the n x k Jacobian
    ll, gr, gm = lib.loglik_grad_batch_mean(X, y, J, L, A, N, kid_of(lib, kernel))
    for s in range(4):
        post = O.posterior_fit(X, y, L[s], A[s], N[s], kernel)
        ref = J @ post.alpha_w
        assert np.max(np.abs(gm[s] - ref)) <= TOL_LL * np.linalg.norm(ref)


# ---- x-gradients -------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("kernel", KERNELS, ids=IDS)
def test_predict_grad_and_ei_value_grad(lib, kernel):
    X, Y, ls, amp, ns, gp, post = _fit(lib, kernel, 200, 4, seed=31)
    Xs = np.random.default_rng(32).random((4, 256))
    Xs[:, :4] = X[:, 10:14]                     # exactly on training points (Matern12: the r = 0 convention)
    mu, var, dmu, dvar, st = lib.gp_predict_grad([gp], 1, 1, Xs)
    rmu, rvar, rdmu, rdvar, rst = O.mean_var_grad(post, Xs)
    assert np.all(np.isfinite(dmu)) and np.all(np.isfinite(dvar))
    assert _close(mu[0], rmu, TOL_POST)
    for j in range(4):
        assert _close(dmu[0, j], rdmu[j], 1e-8, scale=np.max(np.abs(rdmu)))
        assert _close(dvar[0, j], rdvar[j], 1e-8, scale=np.max(np.abs(rdvar)))
    best = float(np.quantile(Y[0], 0.8))
    val, grad = lib.ei_value_grad([gp], 1, 1, Xs, [1.0], best, None)
    rv, rg = O.ei_value_grad([post], Xs, [1.0], best, None)
    assert np.all(np.isfinite(grad))
    assert _close(val, rv, TOL_POST)
    assert _close(grad, rg, 1e-8, scale=np.max(np.abs(rg)))
    gp.free()


@pytest.mark.parametrize("kernel", KERNELS, ids=IDS)
def test_mcei_value_grad(lib, kernel):
    X, Y, ls, amp, ns, gp, post = _fit(lib, kernel, 150, 3, seed=41)
    Xs = np.random.default_rng(42).random((3, 200))
    Xs[:, 0] = X[:, 5]
    eps = np.random.default_rng(43).standard_normal((1, 64))
    best = float(np.quantile(Y[0], 0.7))
    val, grad = lib.mcei_value_grad([gp], 1, 1, Xs, 1, eps, best, None, c0=0.0, c=[1.0])
    saved = MO.O
    MO.O = O                                     # the reference's posterior maths with the new kernels
    try:
        rv, rg = MO.mc_ei_value_grad([[post]], Xs, 1, 0.0, np.array([1.0]), np.zeros(1), np.zeros(1), eps, best, None)
    finally:
        MO.O = saved
    assert np.all(np.isfinite(grad))
    assert _close(val, rv, TOL_POST)
    assert _close(grad, rg, 1e-8, scale=np.max(np.abs(rg)))
    gp.free()


# ---- EI scoring, screening, top-k, device candidates -------------------------------------------------------------

@pytest.mark.parametrize("kernel", KERNELS, ids=IDS)
def test_ei_score_matches_oracle(lib, kernel):
    X, Y, ls, amp, ns, gp, post = _fit(lib, kernel, 300, 5, seed=51)
    Xs = np.random.default_rng(52).random((5, 5000))
    best = float(np.max(Y[0]))
    acq, bv, bi = lib.ei_score([gp], 1, 1, Xs, [1.0], best, None)
    ref, _, _ = O.ei_acquisition([[post]], Xs, [1.0], best, None)
    m = ref > 1e-200
    assert np.max(np.abs(acq[m] - ref[m]) / ref[m]) <= TOL_POST
    assert bi == O.julia_argmax_fast(ref)
    gp.free()


@pytest.fixture(scope="module")
def big(lib):
    X, Y, ls, amp, ns = make_problem(2048, 8, seed=61)
    Xs = np.random.default_rng(62).random((8, 200_000))
    return X, Y, ls, amp, ns, Xs


@pytest.mark.parametrize("kernel", KERNELS, ids=IDS)
def test_screened_argmax_and_topk_bitwise(lib, big, kernel, monkeypatch):
    X, Y, ls, amp, ns, Xs = big
    best = float(np.max(Y[0]))
    ref5 = lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], 2)
    monkeypatch.setenv("BOSS_SCREEN_F64", "1")
    lib.ei_score([ref5], 1, 1, Xs, [1.0], best, None, want_acq=False)
    amb_f64 = lib.dbg_screen_ambiguous()
    monkeypatch.delenv("BOSS_SCREEN_F64")
    ref5.free()
    gp = lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], kid_of(lib, kernel))
    _, bv, bi = lib.ei_score([gp], 1, 1, Xs, [1.0], best, None, want_acq=False)
    assert lib.dbg_screen_stats()[0] == 1
    amb = lib.dbg_screen_ambiguous()
    assert amb[0] == amb_f64[0] == 0                       # no ambiguous band: the FP32 tier did not run
    acq, bv0, bi0 = lib.ei_score([gp], 1, 1, Xs, [1.0], best, None)   # acq output: never screened
    monkeypatch.setenv("BOSS_NO_SCREEN", "1")
    _, bv1, bi1 = lib.ei_score([gp], 1, 1, Xs, [1.0], best, None, want_acq=False)
    monkeypatch.delenv("BOSS_NO_SCREEN")
    assert (bv, bi) == (bv1, bi1) == (bv0, bi0)
    k = 64
    tv, ti = lib.ei_score_topk([gp], 1, 1, Xs, [1.0], best, None, k)
    order = np.lexsort((np.arange(acq.size), -acq))[:k]
    assert np.array_equal(ti, order) and np.array_equal(tv, acq[order])
    gp.free()


@pytest.mark.parametrize("kernel", KERNELS, ids=IDS)
def test_grid_and_uniform_candidates(lib, kernel):
    X, Y, ls, amp, ns, gp, post = _fit(lib, kernel, 100, 2, seed=71)
    best = float(np.max(Y[0]))
    lo, step, cnt = np.zeros(2), np.array([0.01, 0.02]), np.array([101, 51])
    acq, bv, bi, bx = lib.ei_score_grid([gp], 1, 1, lo, step, cnt, [1.0], best, None, want_acq=True)
    g0, g1 = np.meshgrid(lo[0] + step[0] * np.arange(cnt[0]), lo[1] + step[1] * np.arange(cnt[1]), indexing="ij")
    G = np.stack([g0.ravel(), g1.ravel()])
    ref, _, _ = lib.ei_score([gp], 1, 1, G, [1.0], best, None)
    assert np.array_equal(np.sort(acq), np.sort(ref))
    assert bv == np.max(ref)
    lb, ub = np.zeros(2), np.ones(2)
    acq_u, bvu, biu, bxu = lib.ei_score_uniform([gp], 1, 1, 7, 20000, lb, ub, [1.0], best, None, want_acq=True)
    U = lib.uniform_candidates(7, 0, 20000, lb, ub)
    ref_u, bvr, bir = lib.ei_score([gp], 1, 1, U, [1.0], best, None)
    assert np.array_equal(acq_u, ref_u) and (bvu, biu) == (bvr, bir)
    gp.free()


# ---- multi-start drivers -----------------------------------------------------------------------------------------

@pytest.mark.parametrize("kernel", KERNELS, ids=IDS)
def test_multistart_best_is_a_fresh_score(lib, kernel):
    X, Y, ls, amp, ns, gp, post = _fit(lib, kernel, 300, 4, seed=81)
    best = float(np.quantile(Y[0], 0.9))
    starts = np.random.default_rng(82).random((4, 1024))
    lb, ub = np.zeros(4), np.ones(4)
    Xo, fo, bx, bv, bi, _ = lib.ei_maximize_multistart([gp], 1, 1, starts, [1.0], best, None, lb, ub, iters=20)
    acq, _, _ = lib.ei_score([gp], 1, 1, bx[:, None], [1.0], best, None)
    assert np.isfinite(bv) and bv == acq[0]
    eps = np.random.default_rng(83).standard_normal((1, 32))
    Xo, fo, bx, bv, bi, _ = lib.mcei_maximize_multistart([gp], 1, 1, starts, 1, eps, best, None, lb, ub, c0=0.0, c=[1.0],
                                                          iters=20)
    acq, _, _ = lib.mcei_score([gp], 1, 1, bx[:, None], 1, eps, best, None, c0=0.0, c=[1.0])
    assert np.isfinite(bv) and bv == acq[0]
    gp.free()


# ---- append, cov, RQ -> SE ---------------------------------------------------------------------------------------

@pytest.mark.parametrize("kernel", KERNELS, ids=IDS)
def test_append_matches_refit_and_cov(lib, kernel):
    X, Y, ls, amp, ns = make_problem(128, 3, seed=91)       # the append crosses a 128-block boundary
    kid = kid_of(lib, kernel)
    gp = lib.gp_fit(X[:, :127], Y[0, :127], ls[0], amp[0], ns[0], kid)
    for j in (127,):
        assert lib.gp_append(gp, X[:, j], Y[0, j])
    x_new = np.array([0.3, 0.6, 0.1])
    assert lib.gp_append(gp, x_new, 0.25)
    X2, y2 = np.column_stack([X, x_new]), np.append(Y[0], 0.25)
    full = lib.gp_fit(X2, y2, ls[0], amp[0], ns[0], kid)
    Xs = np.random.default_rng(92).random((3, 300))
    a, b = lib.gp_predict(gp, Xs), lib.gp_predict(full, Xs)
    assert _close(a[0], b[0], 1e-9) and _close(a[1], b[1], 1e-9, scale=amp[0] ** 2)
    assert gp.loglik == pytest.approx(full.loglik, rel=1e-9)
    post = O.posterior_fit(X2, y2, ls[0], amp[0], ns[0], kernel)
    mu, cov, rc = lib.gp_cov(full, Xs[:, :40])
    rmu = O.mean_and_var(post, Xs[:, :40])[0]
    rcov = O.posterior_cov(post, Xs[:, :40])[0]
    assert rc == 0
    assert _close(mu, rmu, TOL_POST) and _close(cov, rcov, TOL_POST, scale=amp[0] ** 2)
    gp.free()
    full.free()


def test_rq_large_a_is_se(lib):
    X, Y, ls, amp, ns = make_problem(300, 4, seed=95)
    rq = lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], lib.kernel_rational_quadratic(1e8))
    se = lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], 0)
    Xs = np.random.default_rng(96).random((4, 500))
    a, b = lib.gp_predict(rq, Xs), lib.gp_predict(se, Xs)
    assert _close(a[0], b[0], 1e-6) and _close(a[1], b[1], 1e-6)
    rq.free()
    se.free()


# ---- kernel ids ----------------------------------------------------------------------------------------------------

def test_unknown_kernel_ids_are_rejected(lib):
    X, Y, ls, amp, ns = make_problem(30, 2, seed=97)
    L, A, N = make_hyper_samples(4, 2, seed=98)
    for bad in (4, 7, 255, 256 + lib.RQ_SLOTS - 1, 256 + lib.RQ_SLOTS, -1):
        with pytest.raises(lib.BossError, match="kernel_id"):
            lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], bad)
        with pytest.raises(lib.BossError, match="kernel_id"):
            lib.loglik_batch(X, Y[0], L, A, N, bad)


def test_handle_keeps_its_shape_parameter(lib):
    X, Y, ls, amp, ns = make_problem(200, 3, seed=99)
    Xs = np.random.default_rng(100).random((3, 400))
    gp = lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], lib.kernel_rational_quadratic(1.25))
    before = lib.gp_predict(gp, Xs)
    for a in (0.3, 3.0, 11.0, 1.2500000000000002):
        lib.kernel_rational_quadratic(a)
    after = lib.gp_predict(gp, Xs)
    assert np.array_equal(before[0], after[0]) and np.array_equal(before[1], after[1])
    post = O.posterior_fit(X, Y[0], ls[0], amp[0], ns[0], RQ(1.25))
    assert _close(after[0], O.mean_and_var(post, Xs)[0], TOL_POST)
    gp.free()


# ---- guard bands, multi-device -----------------------------------------------------------------------------------

_REDZONE = r'''
import sys, json
import numpy as np
sys.path.insert(0, sys.argv[1])
import boss_b200
from boss_b200 import _lib as lib
from tests.util_problems import make_problem, make_hyper_samples
lib.init(0)
X, Y, ls, amp, ns = make_problem(200, 5, seed=5)
L, A, N = make_hyper_samples(6, 5, seed=6)
Xs = np.random.default_rng(7).random((5, 3000))
for kid in (3, lib.kernel_rational_quadratic(2.0)):
    gp = lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], kid)
    lib.loglik_batch(X, Y[0], L, A, N, kid)
    lib.loglik_grad_batch(X, Y[0], L, A, N, kid)
    lib.loglik_batch(X[:, :20], Y[0, :20], L, A, N, kid)
    lib.ei_score([gp], 1, 1, Xs, [1.0], float(Y[0].max()), None)
    lib.ei_value_grad([gp], 1, 1, Xs[:, :500], [1.0], float(Y[0].max()), None)
    lib.gp_cov(gp, Xs[:, :30])
    lib.gp_append(gp, Xs[:, 0], 0.1)
    gp.free()
bad, nalloc = lib.dbg_check_redzones()
print(json.dumps({"bad": bad, "allocs": nalloc}))
'''


def test_redzones_stay_clean():
    import json
    r = subprocess.run([sys.executable, "-c", _REDZONE, ROOT], env=dict(os.environ, BOSS_DEBUG_REDZONE="1"),
                       capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    j = json.loads(r.stdout.strip().splitlines()[-1])
    assert j["bad"] == 0 and j["allocs"] > 0


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
from tests.util_problems import make_problem, make_hyper_samples
X, Y, ls, amp, ns = make_problem(300, 4, seed=11)
L, A, N = make_hyper_samples(16, 4, seed=12)
Xs = np.random.default_rng(13).random((4, 50000))
res = []
for multi in (False, True):
    if multi:
        lib.init_multi(2)
    else:
        lib.init(0)
    out = []
    for kid in (3, lib.kernel_rational_quadratic(0.5)):
        gp = lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], kid)
        out += [lib.ei_score([gp], 1, 1, Xs, [1.0], float(Y[0].max()), None)[0],
                lib.loglik_grad_batch(X, Y[0], L, A, N, kid)[1], np.array([gp.loglik])]
        gp.free()
    res.append(out)
    lib.shutdown()
for a, b in zip(*res):
    assert np.array_equal(a, b)
print("multi ok")
'''


@pytest.mark.skipif(_n_gpus() < 2, reason="needs >= 2 GPUs")
def test_two_devices_match_one_bit_for_bit():
    r = subprocess.run([sys.executable, "-c", _MULTI, ROOT], capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert r.returncode == 0 and "multi ok" in r.stdout, r.stdout + r.stderr


# ---- host mirror ---------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("which", ["exp", "rq"])
def test_host_mirror_bo_iteration(lib, which):
    import boss_b200 as B
    kern = B.ExponentialKernel() if which == "exp" else B.RationalQuadraticKernel(2.0)
    rng = np.random.default_rng(3)
    f = lambda x: np.array([np.sin(x[0]) + 0.5 * np.cos(2 * x[1])])
    dom = B.Domain(([0.0, 0.0], [10.0, 10.0]))
    X = B.generate_LHC(dom.bounds, 20, rng)
    Y = np.stack([f(X[:, j]) for j in range(20)], axis=1)

    def problem():
        model = B.GaussianProcess(kernel=kern, lengthscale_priors=[B.mvlognormal([0.5, 0.5], [0.5, 0.5])],
                                  amplitude_priors=[B.LogNormal(0.0, 0.5)], noise_std_priors=[B.Dirac(0.1)])
        return B.BossProblem(f, dom, B.ExpectedImprovement(B.LinFitness([1.0])), model, B.ExperimentData(X, Y))

    for fitter, am in ((B.SamplingMAP(32, seed=1), B.SamplingAM(None, 500, seed=1)),
                       (B.OptimizationMAP(multistart=4, iters=10, seed=0), B.OptimizationAM(multistart=16, iters=10,
                                                                                           seed=0))):
        prob = problem()
        B.bo(prob, fitter, am, B.IterLimit(1))
        assert len(prob.data) == 21 and prob.consistent and np.isfinite(prob.params.loglike)
