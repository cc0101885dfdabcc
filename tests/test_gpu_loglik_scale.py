"""The batched log-likelihood, its hyper-parameter gradient, its prior-mean gradient (alpha^T J) and the batched fit at
the sizes they run at: eight and more row blocks (the separate SYRK -> potrf_tile -> chol_panel diagonal step, the
multi-block triangular inverse, kinv_wtw_kernel and loglik_grad_tile_kernel), every covariance function and padded
input width, 1-16 stream groups, several workspace windows, failed samples on group and window boundaries, and the
device-pointer entry points.

The FP64 oracle is the reference (tests/loglik_scale_oracle.py; its own error against a long-double evaluation is
measured by tests/test_loglik_scale_host.py).  It runs on a few samples per batch only; every other sample is checked
through bit-identity with calls that do not share its window or group.

Runs in about six minutes on one B200, CPU references included.  Peak device memory is about 50 GB: the 33 GB
gradient workspace of n = 4096 (kept by the library's context) plus about 13 GB of handles from the batched fit that
crosses a window at n = 100.
"""
import hashlib

import numpy as np
import pytest

from oracle import boss_oracle as OB
from tests import loglik_scale_oracle as LS
from tests.kernels_more_oracle import KERNEL_MATERN12, RQ
from tests.util_problems import make_hyper_samples, make_problem

pytestmark = pytest.mark.gpu

ALL_KERNELS = [OB.KERNEL_SE, OB.KERNEL_MATERN32, OB.KERNEL_MATERN52, KERNEL_MATERN12, RQ(0.5), RQ(2.0), RQ(50.0)]
IDS = ["se", "matern32", "matern52", "matern12", "rq0.5", "rq2", "rq50"]
WORST = {}


def kid_of(lib, kernel):
    return lib.kernel_rational_quadratic(kernel.a) if isinstance(kernel, RQ) else kernel


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def _same(a, b):
    return np.array_equal(_bits(a), _bits(b))


def _note(family, ratio):
    WORST[family] = max(WORST.get(family, 0.0), float(ratio))
    assert ratio <= 1.0, (family, ratio)


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    for k, v in sorted(WORST.items()):
        print(f"worst ratio to tolerance, {k}: {v:.3g}")


def _jac(X, S=None, seed=0):
    """Prior-mean Jacobian (k = 3, n): shared, or (S, 3, n) per sample."""
    J = np.stack([np.ones(X.shape[1]), X[0], X[-1] ** 2])
    if S is None:
        return J
    return J[None] * (1.0 + 0.1 * np.arange(S))[:, None, None] + 0.01 * np.random.default_rng(seed).random((S, 3, X.shape[1]))


def _check_ref(family, X, Y, J, L, A, N, kernel, samples, ll, gr, gm, mask=None):
    """ll / gr / gm (batch outputs) against the oracle on the given samples; Y (n,) or (S, n), J (k, n) or (S, k, n)."""
    Om = LS.oracle_for(kernel)
    for s in samples:
        y = Y if Y.ndim == 1 else Y[s]
        rl, rg = LS.reference_grad(X, y, L[s], A[s], N[s], kernel, mask)
        _note(f"{family}: value", LS.rel_ratio(ll[s], rl))
        if gr is not None:
            assert np.all(np.isfinite(gr[s]))
            _note(f"{family}: gradient", LS.grad_ratio(gr[s], rg))
        if gm is not None:
            alpha = Om.posterior_fit(X, y, L[s], A[s], N[s], kernel, mask).alpha_w
            ref = (J if J.ndim == 2 else J[s]) @ alpha
            _note(f"{family}: alpha-Jacobian", LS.grad_ratio(gm[s], ref, LS.TOL_JAC))


def _all_modes(lib, X, Y, J, L, A, N, kid, mask=None):
    ll = lib.loglik_batch(X, Y, L, A, N, kid, mask)
    ll_g, gr = lib.loglik_grad_batch(X, Y, L, A, N, kid, mask)
    ll_m, gr_m, gm = lib.loglik_grad_batch_mean(X, Y, J, L, A, N, kid, mask)
    return ll, ll_g, gr, ll_m, gr_m, gm


# ---- 1. reference parity at eight and more blocks ------------------------------------------------------------------

@pytest.mark.parametrize("kernel", ALL_KERNELS, ids=IDS)
def test_bench_shape_every_kernel(lib, kernel):
    """n = 2048, d = 8, S = 10: 16 blocks, 4 stream groups of 3/3/3/1."""
    n, d, S = 2048, 8, 10
    X, Y, _, _, _ = make_problem(n, d, seed=2048)
    L, A, N = make_hyper_samples(S, d, seed=2049)
    Yp = Y[0][None, :] + 0.05 * np.sin(np.arange(S))[:, None]
    kid = kid_of(lib, kernel)
    assert [g[1] for g in LS.window_plan(n, d, S, "grad")["windows"][0]["groups"]] == [3, 3, 3, 1]
    for J in (_jac(X), _jac(X, S, seed=3)):
        Yc = Y[0] if J.ndim == 2 else Yp
        ll, ll_g, gr, ll_m, gr_m, gm = _all_modes(lib, X, Yc, J, L, A, N, kid)
        assert _same(ll, ll_g) and _same(ll, ll_m) and _same(gr, gr_m)
        _check_ref("bench shape", X, Yc, J, L, A, N, kernel, (0, 3, 8, 9) if J.ndim == 2 else (3, 9), ll, gr, gm)
        for s in range(S):
            one = _all_modes(lib, X, Yc if Yc.ndim == 1 else Yc[s:s + 1], J if J.ndim == 2 else J[s:s + 1],
                             L[s:s + 1], A[s:s + 1], N[s:s + 1], kid)
            for a, b in zip((ll, ll_g, gr, ll_m, gr_m, gm), one):
                assert _same(a[s:s + 1], b), s


# (n, d, kernel, options): n = 769 / 1000 / 2047 leave 1 / 104 / 127 real rows in the last block; every padded width
# DP in {2, 4, 6, 8, 12, 16, 32}; every kernel id at DP = 32.
SHAPES = [(769, 2, OB.KERNEL_SE, ""), (769, 32, KERNEL_MATERN12, ""), (769, 32, OB.KERNEL_MATERN52, "mask"),
          (1000, 4, OB.KERNEL_MATERN32, ""), (1000, 32, RQ(2.0), "per_sample_y"), (1000, 16, OB.KERNEL_MATERN52, ""),
          (1000, 32, OB.KERNEL_MATERN32, ""), (2047, 6, RQ(50.0), ""), (2047, 32, OB.KERNEL_SE, ""),
          (2047, 12, RQ(0.5), ""), (2047, 8, KERNEL_MATERN12, "")]


@pytest.mark.parametrize("n,d,kernel,opt", SHAPES)
def test_every_padding_class_at_eight_blocks_and_more(lib, n, d, kernel, opt):
    S = 3
    X, Y, _, _, _ = make_problem(n, d, seed=n + d)
    L, A, N = make_hyper_samples(S, d, seed=n + d + 1)
    mask = None
    if opt == "mask":
        mask = np.zeros(d, bool); mask[[1, 7, 30]] = True
        X[mask] = np.round(X[mask] * 5)
    Yc = Y[0][None, :] * np.array([1.0, 0.5, -1.0])[:, None] if opt == "per_sample_y" else Y[0]
    J = _jac(X)
    ll, ll_g, gr, ll_m, gr_m, gm = _all_modes(lib, X, Yc, J, L, A, N, kid_of(lib, kernel), mask)
    assert _same(ll, ll_g) and _same(ll, ll_m) and _same(gr, gr_m)
    _check_ref("padding classes", X, Yc, J, L, A, N, kernel, (0, 2), ll, gr, gm, mask)


def test_matern12_duplicates_across_blocks(lib):
    n, d, S = 1000, 3, 3
    X, Y, _, _, _ = make_problem(n, d, seed=12)
    X[:, 900] = X[:, 5]; X[:, 777] = X[:, 130]; X[:, 999] = X[:, 998]
    L, A, N = make_hyper_samples(S, d, seed=13)
    ll, gr = lib.loglik_grad_batch(X, Y[0], L, A, N, KERNEL_MATERN12)
    assert np.all(np.isfinite(gr)) and np.all(np.isfinite(ll))
    _check_ref("matern12 duplicates", X, Y[0], None, L, A, N, KERNEL_MATERN12, range(S), ll, gr, None)


# ---- 2. long-double adjudication at eight blocks -------------------------------------------------------------------

@pytest.mark.parametrize("kernel", [OB.KERNEL_MATERN52, KERNEL_MATERN12, RQ(2.0)], ids=["matern52", "matern12", "rq2"])
def test_gradient_as_close_to_long_double_truth_as_the_oracle(lib, kernel):
    n, d = 1000, 6
    X, Y, _, _, _ = make_problem(n, d, seed=1000)
    L, A, N = make_hyper_samples(1, d, seed=1001)
    ll_t, g_t = LS.adjudicator_grad_longdouble(X, Y[0], L[0], A[0], N[0], kernel)
    ll_o, g_o = LS.reference_grad(X, Y[0], L[0], A[0], N[0], kernel)
    ll_g, g_g = lib.loglik_grad_batch(X, Y[0], L, A, N, kid_of(lib, kernel))
    e_o, e_g = np.max(np.abs(g_o - g_t)), np.max(np.abs(g_g[0] - g_t))
    bound = max(4 * e_o, 1e-11 * np.linalg.norm(g_t))
    print(f"{kernel}: |g_gpu - g_ld| = {e_g:.3g}, |g_oracle - g_ld| = {e_o:.3g}, |g| = {np.linalg.norm(g_t):.3g}")
    _note("long-double gradient", e_g / bound)
    _note("long-double value", abs(ll_g[0] - ll_t) / max(4 * abs(ll_o - ll_t), 1e-12 * abs(ll_t)))


# ---- 3. stream groups ----------------------------------------------------------------------------------------------

def _fit_sig(lib, g, Xs):
    Lf, Wf, al = lib.dbg_factors(g)
    mu, var, _ = lib.gp_predict(g, Xs)
    h = hashlib.sha256()
    for a in (Lf, Wf, al, mu, var, [g.loglik]):
        h.update(_bits(a).tobytes())
    return h.hexdigest()


def test_stream_groups_are_bit_identical(lib, monkeypatch):
    n, d, S = 900, 4, 37
    X, Y, _, _, _ = make_problem(n, d, seed=900)
    L, A, N = make_hyper_samples(S, d, seed=901)
    Yp = Y[0][None, :] + 0.1 * np.cos(np.arange(S))[:, None]
    J = _jac(X, S, seed=902)
    Xs = np.random.default_rng(903).random((d, 500))
    kid = OB.KERNEL_MATERN52

    def run():
        ll, gr = lib.loglik_grad_batch(X, Yp, L, A, N, kid)
        out = (lib.loglik_batch(X, Yp, L, A, N, kid), ll, gr, *lib.loglik_grad_batch_mean(X, Yp, J, L, A, N, kid))
        gps = lib.gp_fit_batch(X, Yp, L, A, N, kid)
        sig = [_fit_sig(lib, g, Xs) for g in gps]
        lls = np.array([g.loglik for g in gps])
        for g in gps:
            g.free()
        return out, sig, lls

    monkeypatch.delenv("BOSS_LL_GROUPS", raising=False)
    base, base_sig, base_ll = run()
    assert _same(base_ll, base[0])
    edges = set(LS.boundary_samples(LS.window_plan(n, d, S, "grad")))
    configs = [(g, False) for g in (1, 2, 3, 4, 5, 16)] + [(None, True)]
    for groups, timing in configs:
        edges.update(LS.boundary_samples(LS.window_plan(n, d, S, "grad", groups=groups, timing=timing)))
        if groups is None:
            monkeypatch.delenv("BOSS_LL_GROUPS", raising=False)
        else:
            monkeypatch.setenv("BOSS_LL_GROUPS", str(groups))
        lib.set_timing(timing)
        try:
            out, sig, _ = run()
        finally:
            lib.set_timing(False)
        for a, b in zip(base, out):
            assert _same(a, b), (groups, timing)
        assert sig == base_sig, (groups, timing)
    monkeypatch.delenv("BOSS_LL_GROUPS", raising=False)
    edges = sorted(edges)
    _check_ref("stream groups", X, Yp, J, L, A, N, kid, edges, base[1], base[2], base[5])
    gps = lib.gp_fit_batch(X, Yp, L, A, N, kid)
    for s in edges:
        single = lib.gp_fit(X, Yp[s], L[s], A[s], N[s], kid)
        post = OB.posterior_fit(X, Yp[s], L[s], A[s], N[s], kid)
        mu, var, _ = lib.gp_predict(gps[s], Xs)
        for mr, vr in (lib.gp_predict(single, Xs)[:2], OB.mean_and_var(post, Xs)[:2]):
            _note("stream groups: posterior", max(float(np.max(np.abs(mu - mr) / np.abs(mr))),
                                                  float(np.max(np.abs(var - vr) / np.abs(vr)))) / LS.TOL_POST)
        single.free()
    for g in gps:
        g.free()


# ---- 4. workspace windows ------------------------------------------------------------------------------------------

def _launches(lib, f):
    c0 = lib.launch_count()
    r = f()
    return lib.launch_count() - c0, r


def _window_problem(n, d, S, seed):
    X, Y, _, _, _ = make_problem(n, d, seed=seed)
    L, A, N = make_hyper_samples(S, d, seed=seed + 1)
    Yp = Y[0][None, :] + 0.2 * np.sin(0.001 * np.arange(S))[:, None]
    return X, Yp, L, A, N


def _oracle_samples(S, Sb, n_random, seed):
    rng = np.random.default_rng(seed)
    return sorted({0, Sb - 1, Sb, S - 1, *rng.integers(0, S, n_random).tolist()})


def _chunks(S, step):
    return [(a, min(S, a + step)) for a in range(0, S, step)]


def test_value_across_a_window(lib):
    n, d, S = 100, 3, 32768 + 5
    plan = LS.window_plan(n, d, S, "value")
    Sb = plan["Sb"]
    assert Sb == 32768 and len(plan["windows"]) == 2
    X, Yp, L, A, N = _window_problem(n, d, S, seed=100)
    kid = OB.KERNEL_MATERN32
    f = lambda a, b: lib.loglik_batch(X, Yp[a:b], L[a:b], A[a:b], N[a:b], kid)
    nl, ll = _launches(lib, lambda: f(0, S))
    nl_sb, _ = _launches(lib, lambda: f(0, Sb))
    nl_rest, _ = _launches(lib, lambda: f(Sb, S))
    assert nl - nl_sb == nl_rest > 0                    # the batch ran as a window of Sb and one of S - Sb
    for a, b in _chunks(S, 10000):                      # chunks that do not line up with the window
        assert _same(ll[a:b], f(a, b)), (a, b)
    for s in _oracle_samples(S, Sb, 60, 7):
        _note("window: value", LS.rel_ratio(ll[s], OB.gp_loglik(X, Yp[s], L[s], A[s], N[s], kid)))


def test_gradients_across_a_window(lib):
    n, d, S = 100, 3, 32773
    plan = LS.window_plan(n, d, S, "grad")
    Sb = plan["Sb"]
    assert Sb == 32768 and len(plan["windows"]) == 2
    X, Yp, L, A, N = _window_problem(n, d, S, seed=200)
    J = _jac(X, S, seed=201)
    kid = OB.KERNEL_MATERN52
    g = lambda a, b: lib.loglik_grad_batch(X, Yp[a:b], L[a:b], A[a:b], N[a:b], kid)
    m = lambda a, b: lib.loglik_grad_batch_mean(X, Yp[a:b], J[a:b], L[a:b], A[a:b], N[a:b], kid)
    for fn, name in ((g, "gradient"), (m, "mean-gradient")):
        nl, full = _launches(lib, lambda: fn(0, S))
        nl_sb, _ = _launches(lib, lambda: fn(0, Sb))
        nl_rest, _ = _launches(lib, lambda: fn(Sb, S))
        assert nl - nl_sb == nl_rest > 0, name
        for a, b in _chunks(S, 10000):
            part = fn(a, b)
            for x, y in zip(full, part):
                assert _same(x[a:b], y), (name, a, b)
        if name == "gradient":
            ll, gr = full
        else:
            assert _same(full[0], ll) and _same(full[1], gr)
            gm = full[2]
    _check_ref("window n=100", X, Yp, J, L, A, N, kid, _oracle_samples(S, Sb, 60, 8), ll, gr, gm)


def test_gradient_across_a_window_at_n4096(lib):
    """per = 3 n_pad^2 8 + 2 nblk 128^2 8 = 411 041 792 B: Sb = 83, a window of 4 groups (21/21/21/20), then 7."""
    n, d, S = 4096, 4, 90
    plan = LS.window_plan(n, d, S, "grad")
    Sb = plan["Sb"]
    assert Sb == 83 and [w["ngroups"] for w in plan["windows"]] == [4, 1]
    X, Yp, L, A, N = _window_problem(n, d, S, seed=4096)
    kid = OB.KERNEL_SE
    g = lambda a, b: lib.loglik_grad_batch(X, Yp[a:b], L[a:b], A[a:b], N[a:b], kid)
    nl, (ll, gr) = _launches(lib, lambda: g(0, S))
    nl_sb, _ = _launches(lib, lambda: g(0, Sb))
    nl_rest, _ = _launches(lib, lambda: g(Sb, S))
    assert nl - nl_sb == nl_rest > 0
    for a, b in ((0, 45), (45, 90)):
        pl, pg = g(a, b)
        assert _same(ll[a:b], pl) and _same(gr[a:b], pg), (a, b)
    _check_ref("window n=4096", X, Yp, None, L, A, N, kid, (0, Sb - 1, Sb, S - 1), ll, gr, None)


def test_fit_batch_across_a_window(lib):
    n, d, S = 100, 3, 32770
    Sb = LS.window_plan(n, d, S, "fit")["Sb"]
    assert Sb == 32768
    X, Yp, L, A, N = _window_problem(n, d, S, seed=300)
    kid = OB.KERNEL_MATERN52
    Xs = np.random.default_rng(301).random((d, 500))
    ll = lib.loglik_batch(X, Yp, L, A, N, kid)
    nl, gps = _launches(lib, lambda: lib.gp_fit_batch(X, Yp, L, A, N, kid))
    picks = (0, Sb - 1, Sb, S - 1)
    sig = {}
    try:
        assert all(g is not None for g in gps)
        for s in picks:
            one = lib.gp_fit_batch(X, Yp[s:s + 1], L[s:s + 1], A[s:s + 1], N[s:s + 1], kid)[0]
            sig[s] = _fit_sig(lib, gps[s], Xs)
            assert sig[s] == _fit_sig(lib, one, Xs), s
            assert gps[s].loglik == one.loglik == ll[s]
            _note("window fit: loglik", LS.rel_ratio(gps[s].loglik, OB.gp_loglik(X, Yp[s], L[s], A[s], N[s], kid)))
            post = OB.posterior_fit(X, Yp[s], L[s], A[s], N[s], kid)
            mu, var, _ = lib.gp_predict(gps[s], Xs)
            mr, vr, _ = OB.mean_and_var(post, Xs)
            _note("window fit: posterior", max(float(np.max(np.abs(mu - mr) / np.abs(mr))),
                                               float(np.max(np.abs(var - vr) / np.abs(vr)))) / LS.TOL_POST)
            one.free()
        assert np.array_equal(np.array([g.loglik for g in gps]), ll)
    finally:
        for g in gps:
            if g is not None:
                g.free()
        del gps
    nl_sb, gps = _launches(lib, lambda: lib.gp_fit_batch(X, Yp[:Sb], L[:Sb], A[:Sb], N[:Sb], kid))
    for g in gps:
        g.free()
    del gps
    nl_rest, gps = _launches(lib, lambda: lib.gp_fit_batch(X, Yp[Sb:], L[Sb:], A[Sb:], N[Sb:], kid))
    for g in gps:
        g.free()
    assert nl - nl_sb == nl_rest > 0


# ---- 5. failed samples on group and window boundaries -------------------------------------------------------------

def _with_failures(n, d, S, bad, seed, same=40):
    """The first `same` training points coincide; samples in `bad` get amplitude 1e6 and noise 0, so their K holds a
    block of a^2 with nothing on its diagonal to keep it positive definite (test_fit_batch_reports_non_pd_samples)."""
    X, Yp, L, A, N = _window_problem(n, d, S, seed)
    X[:, :same] = X[:, :1]
    A = A.copy(); N = N.copy()
    A[bad] = 1e6
    N[bad] = 0.0
    return X, Yp, L, A, N


@pytest.mark.parametrize("n,S,bad", [(900, 37, [9, 10, 36]), (100, 32770, [0, 32767, 32768])],
                         ids=["group_edges", "window_edge"])
def test_failed_samples_on_boundaries(lib, n, S, bad):
    """Non-PD samples first / last in a group (n = 900: groups 10/10/10/7) and on both sides of a window (n = 100)."""
    d, kid = 3, OB.KERNEL_MATERN52
    X, Yp, L, A, N = _with_failures(n, d, S, bad, seed=n + 5)
    J = _jac(X, S, seed=n)
    keep = np.setdiff1d(np.arange(S), bad)
    for mode in ("value", "grad"):
        assert set(bad) <= set(LS.boundary_samples(LS.window_plan(n, d, S, mode))), mode
    ll = lib.loglik_batch(X, Yp, L, A, N, kid)
    ll_g, gr = lib.loglik_grad_batch(X, Yp, L, A, N, kid)
    ll_m, gr_m, gm = lib.loglik_grad_batch_mean(X, Yp, J, L, A, N, kid)
    assert np.all(ll[bad] == -np.inf) and np.all(ll_g[bad] == -np.inf) and np.all(ll_m[bad] == -np.inf)
    assert np.all(gr[bad] == 0.0) and np.all(gr_m[bad] == 0.0) and np.all(gm[bad] == 0.0)
    assert np.all(np.isfinite(ll[keep]))
    sub = (X, Yp[keep], L[keep], A[keep], N[keep], kid)
    assert _same(ll[keep], lib.loglik_batch(*sub))
    r = lib.loglik_grad_batch(*sub)
    assert _same(ll_g[keep], r[0]) and _same(gr[keep], r[1])
    r = lib.loglik_grad_batch_mean(X, Yp[keep], J[keep], *sub[2:])
    assert _same(ll_m[keep], r[0]) and _same(gr_m[keep], r[1]) and _same(gm[keep], r[2])
    if S < 1000:
        gps = lib.gp_fit_batch(X, Yp, L, A, N, kid)
        assert all(gps[b] is None for b in bad) and all(gps[s] is not None for s in keep)
        assert np.array_equal(np.array([gps[s].loglik for s in keep]), ll[keep])
        for g in gps:
            if g is not None:
                g.free()


def test_fit_batch_failures_on_both_sides_of_a_window(lib):
    n, d, S = 100, 3, 32770
    bad = [32767, 32768]
    X, Yp, L, A, N = _with_failures(n, d, S, bad, seed=400)
    kid = OB.KERNEL_MATERN52
    Xs = np.random.default_rng(401).random((d, 200))
    ll = lib.loglik_batch(X, Yp, L, A, N, kid)
    gps = lib.gp_fit_batch(X, Yp, L, A, N, kid)
    try:
        assert gps[32767] is None and gps[32768] is None
        assert sum(g is None for g in gps) == 2
        for s in (0, 32766, 32769):
            one = lib.gp_fit_batch(X, Yp[s:s + 1], L[s:s + 1], A[s:s + 1], N[s:s + 1], kid)[0]
            assert _fit_sig(lib, gps[s], Xs) == _fit_sig(lib, one, Xs) and gps[s].loglik == ll[s]
            one.free()
    finally:
        for g in gps:
            if g is not None:
                g.free()


# ---- 6. device-pointer entry points --------------------------------------------------------------------------------

def _dev_calls(lib, torch, X, Y, L, A, N, kid, stream=None, prep=None):
    """loglik_batch_dev and loglik_grad_batch_dev on device copies of the inputs; prep(tensors) may rewrite them on
    `stream` before the calls."""
    n, d = X.shape[1], X.shape[0]
    S = L.shape[0]
    t = [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (X.T, Y, L, A, N)]
    if prep is not None:
        t = prep(t)
    ldy = 0 if Y.ndim == 1 else n
    out = torch.empty(S, dtype=torch.float64, device="cuda")
    out_g = torch.empty(S, dtype=torch.float64, device="cuda")
    grad = torch.empty((S, d + 2), dtype=torch.float64, device="cuda")
    ptr = [x.data_ptr() for x in t]
    lib.loglik_batch_dev(ptr[0], d, n, ptr[1], ldy, ptr[2], ptr[3], ptr[4], kid, S, out.data_ptr(), stream=stream)
    lib.loglik_grad_batch_dev(ptr[0], d, n, ptr[1], ldy, ptr[2], ptr[3], ptr[4], kid, S, out_g.data_ptr(),
                              grad.data_ptr(), stream=stream)
    torch.cuda.synchronize()
    return out.cpu().numpy(), out_g.cpu().numpy(), grad.cpu().numpy()


@pytest.mark.parametrize("n,S,shared_y", [(900, 12, True), (900, 12, False), (100, 32769, False)],
                         ids=["shared_y", "per_sample_y", "window"])
def test_dev_entry_points_equal_the_host_calls(lib, n, S, shared_y):
    torch = pytest.importorskip("torch")
    d, kid = 5, OB.KERNEL_MATERN32
    X, Yp, L, A, N = _window_problem(n, d, S, seed=500 + n)
    Y = Yp[0] if shared_y else Yp
    if n == 100:
        assert len(LS.window_plan(n, d, S, "grad")["windows"]) == 2
    ll, ll_g, gr = _dev_calls(lib, torch, X, Y, L, A, N, kid)
    assert _same(ll, lib.loglik_batch(X, Y, L, A, N, kid))
    h = lib.loglik_grad_batch(X, Y, L, A, N, kid)
    assert _same(ll_g, h[0]) and _same(gr, h[1])


def test_dev_entry_points_wait_for_inputs_made_on_a_side_stream(lib):
    torch = pytest.importorskip("torch")
    n, d, S, kid = 900, 4, 16, OB.KERNEL_MATERN52
    X, Yp, L, A, N = _window_problem(n, d, S, seed=600)
    ref = (lib.loglik_batch(X, Yp, L, A, N, kid), *lib.loglik_grad_batch(X, Yp, L, A, N, kid))
    side = torch.cuda.Stream()

    def late(t):
        """zeroed copies that receive the inputs only at the end of a few milliseconds of work on `side`"""
        bufs = [torch.zeros_like(x) for x in t]
        big = torch.rand((4096, 4096), device="cuda")
        torch.cuda.synchronize()
        with torch.cuda.stream(side):
            for _ in range(20):
                big = big @ big * 1e-3
            for b, x in zip(bufs, t):
                b.copy_(x)
        return bufs

    for _ in range(2):
        got = _dev_calls(lib, torch, X, Yp, L, A, N, kid, stream=side.cuda_stream, prep=late)
        for a, b in zip(got, ref):
            assert _same(a, b)
