"""The posterior, its x-gradients and EI at the sizes they run at, against the FP64 reference: every covariance function
under every scoring path (wide with the fused epilogue, wide with row splits, narrow and quarter, default and forced),
every padded input width, the chunk edges of large calls, Bayesian-inference samples of several outputs, slices of
different block counts in one call, handles grown across a capacity boundary by boss_gp_append, and the single-matrix
fit with the posterior covariance.

The reference is tests/posterior_scale_oracle.py (its distance from a long-double evaluation is measured by
tests/test_posterior_scale_host.py).  At large M it runs on a strided subset of the candidates that always holds the
candidates either side of every chunk boundary and the last one.  Every scoring call checks the paths it took
(boss_dbg_score_paths) against the mirror of the library's dispatch, so a recalibrated cost model cannot silently move a
case off the path it is meant to test.
"""
import numpy as np
import pytest
import scipy.linalg as sl

from oracle import boss_oracle as OB
from tests import posterior_scale_oracle as PS
from tests.kernels_more_oracle import KERNEL_MATERN12, RQ, O as OK
from tests.util_problems import make_problem, relerr

pytestmark = pytest.mark.gpu

KERNELS = [OB.KERNEL_SE, OB.KERNEL_MATERN32, OB.KERNEL_MATERN52, KERNEL_MATERN12, RQ(0.5), RQ(3.0)]
IDS = ["se", "matern32", "matern52", "matern12", "rq0.5", "rq3"]
FORCED = [("wide", False), ("narrow", False), ("quarter", False), (None, True)]
WORST = {}
SEEN = {}   # paths seen under the default dispatch at n >= 2047: (mode) -> set of paths


def kid_of(lib, kernel):
    return lib.kernel_rational_quadratic(kernel.a) if isinstance(kernel, RQ) else kernel


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def _same(a, b):
    return np.array_equal(_bits(a), _bits(b))


def _note(family, r):
    for k, v in r.items():
        WORST[f"{family}: {k}"] = max(WORST.get(f"{family}: {k}", 0.0), float(v))
        assert v <= 1.0, (family, k, v)


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    for k, v in sorted(WORST.items()):
        print(f"worst ratio to tolerance, {k}: {v:.3g}")
    for k, v in sorted(SEEN.items()):
        print(f"paths taken by default at n >= 2047, {k}: {sorted(v)}")


def _env(monkeypatch, path, unfused):
    for k in ("BOSS_SCORE_PATH", "BOSS_UNFUSED_SCORE"):
        monkeypatch.delenv(k, raising=False)
    if path:
        monkeypatch.setenv("BOSS_SCORE_PATH", path)
    if unfused:
        monkeypatch.setenv("BOSS_UNFUSED_SCORE", "1")


def _expect_paths(lib, n_per_slice, M, d, xgrad, pgrad=False, nsl=1, path=None, unfused=False, mode=None):
    plan = PS.score_plan(n_per_slice, M, d, xgrad, pgrad, nsl, path, unfused)
    got = lib.dbg_score_paths()
    assert got == PS.plan_counts(plan), (n_per_slice, M, d, xgrad, path, unfused, got)
    if mode and path is None and not unfused and min(np.atleast_1d(n_per_slice)) >= 2047:
        SEEN.setdefault(mode, set()).update(p["path"] for p in plan["passes"])
    return plan


def _subset(M, plans, k=600):
    """Every candidate when M <= 2000, else k strided ones, the candidates either side of every chunk boundary of
    each plan, and the last."""
    if M <= 2000:
        return np.arange(M)
    s = set(np.linspace(0, M - 1, k).astype(np.int64).tolist())
    for p in plans:
        s.update(PS.chunk_edges(p, M))
    return np.array(sorted(s))


class Ref:
    """FP64 reference posterior and gradients of one GP at the candidates Xs[:, idx]."""

    def __init__(self, kernel, X, y, ls, amp, ns, Xs, idx, mask=None, pm=None, pmg=None):
        Om = PS.reference(kernel)
        self.idx = np.asarray(idx)
        self.pos = {int(m): i for i, m in enumerate(self.idx)}
        Xsub = Xs[:, self.idx]
        self.post = Om.posterior_fit(X, y, ls, amp, ns, kernel, mask)
        self.mu, self.var, self.dmu, self.dvar, self.st = Om.mean_var_grad(
            self.post, Xsub, None if pm is None else pm[self.idx], None if pmg is None else pmg[:, self.idx])
        self.bounds = PS.post_bounds(X, y, ls, amp, ns, kernel, Xsub, mask)
        self.Om, self.Xsub = Om, Xsub

    def at(self, sel):
        p = np.array([self.pos[int(m)] for m in sel])
        return self.mu[p], self.var[p], self.dmu[:, p], self.dvar[:, p]

    def ei(self, best):
        acq = self.Om.ei_acquisition([[self.post]], self.Xsub, [1.0], best, None)[0]
        return acq, self.Om.ei_value_grad([self.post], self.Xsub, [1.0], best, None)[1]

    def check(self, family, sel, mu, var, dmu=None, dvar=None):
        rm, rv, rdm, rdv = self.at(sel)
        r = dict(mu=PS.ratio(mu[sel], rm, PS.TOL_POST, self.bounds[0]), var=PS.ratio(var[sel], rv, PS.TOL_POST, self.bounds[1]))
        if dmu is not None:
            r.update(dmu=PS.grad_ratio(dmu[:, sel], rdm), dvar=PS.grad_ratio(dvar[:, sel], rdv))
        _note(family, r)


# ---- 1. every kernel under every path ------------------------------------------------------------------------------

# M of the value-only and gradient calls, chosen by the mirror so that the default dispatch runs every path at least
# once: quarter (300), wide with row splits (2250 / 1100), wide fused (37888), and a two-chunk call whose tail is narrow
# (value) or quarter (gradient)
PROBLEMS = [(2047, 8, (300, 2250, 37888, 75776 + 300), (300, 2250, 37889)),
            (4096, 4, (300, 1100, 37888, 75777), (300, 1100, 37889))]


@pytest.fixture(scope="module", params=[(k, p) for k in range(len(KERNELS)) for p in range(len(PROBLEMS))],
                ids=[f"{IDS[k]}-n{PROBLEMS[p][0]}" for k in range(len(KERNELS)) for p in range(len(PROBLEMS))])
def kernel_case(request, lib):
    kernel = KERNELS[request.param[0]]
    n, d, vms, gms = PROBLEMS[request.param[1]]
    X, Y, ls, amp, ns = make_problem(n, d, seed=n + 7)
    Mmax = max(vms + gms)
    Xs = np.random.default_rng(n + 8).random((d, Mmax))
    Xs[:, 5] = X[:, 11]                                   # a candidate on a training point
    subs = {}
    for M in set(vms + gms):
        subs[M] = _subset(M, [PS.score_plan(n, M, d, False), PS.score_plan(n, M, d, True)])
    ref = Ref(kernel, X, Y[0], ls[0], amp[0], ns[0], Xs, np.unique(np.concatenate(list(subs.values()))))
    gp = lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], kid_of(lib, kernel))
    assert gp is not None
    best = float(np.quantile(Y[0], 0.9))
    acq_ref, g_ref = ref.ei(best)
    yield dict(kernel=kernel, n=n, d=d, vms=vms, gms=gms, Xs=Xs, subs=subs, ref=ref, gp=gp, best=best, acq_ref=acq_ref,
               g_ref=g_ref)
    gp.free()


def test_every_kernel_and_path(lib, kernel_case, monkeypatch):
    c = kernel_case
    n, d, gp, ref, best = c["n"], c["d"], c["gp"], c["ref"], c["best"]
    fam = f"{IDS[KERNELS.index(c['kernel'])]} n={n}"
    # the default dispatch of these calls runs all four paths without gradients and all but narrow with them
    default = {mode: {p["path"] for M in c[key] for p in PS.score_plan(n, M, d, mode == "gradient")["passes"]}
               for mode, key in (("value", "vms"), ("gradient", "gms"))}
    assert default == dict(value=set(PS.PATHS), gradient={"wide_fused", "wide_split", "quarter"}), default
    for M in c["vms"]:
        Xm, sel = c["Xs"][:, :M], c["subs"][M]
        p = np.array([ref.pos[int(m)] for m in sel])
        base = None
        for path, unfused in [(None, False)] + FORCED:
            _env(monkeypatch, path, unfused)
            mu, var, st = lib.gp_predict(gp, Xm)
            _expect_paths(lib, n, M, d, False, path=path, unfused=unfused, mode="value")
            acq, bv, bi = lib.ei_score([gp], 1, 1, Xm, [1.0], best, None)
            _expect_paths(lib, n, M, d, False, path=path, unfused=unfused)
            if base is None:
                base = (mu, var, acq)
                assert np.all(st == 0)
                ref.check(f"{fam} value", sel, mu, var)
                _note(f"{fam} ei_score", dict(acq=PS.grad_ratio(acq[sel][None], c["acq_ref"][p][None], PS.TOL_POST)))
            else:
                assert _same(mu, base[0]) and _same(var, base[1]) and _same(acq, base[2]), (M, path, unfused)
    for M in c["gms"]:
        Xm, sel = c["Xs"][:, :M], c["subs"][M]
        p = np.array([ref.pos[int(m)] for m in sel])
        base = None
        for path, unfused in [(None, False)] + FORCED:
            _env(monkeypatch, path, unfused)
            mu, var, dmu, dvar, st = lib.gp_predict_grad([gp], 1, 1, Xm)
            _expect_paths(lib, n, M, d, True, pgrad=True, path=path, unfused=unfused, mode="gradient")
            val, g = lib.ei_value_grad([gp], 1, 1, Xm, [1.0], best, None)
            _expect_paths(lib, n, M, d, True, path=path, unfused=unfused)
            if base is None:
                base = (mu, var, dmu, dvar, val, g)
                ref.check(f"{fam} gradient", sel, mu[0], var[0], dmu[0], dvar[0])
                _note(f"{fam} ei_value_grad", dict(val=PS.grad_ratio(val[sel][None], c["acq_ref"][p][None], PS.TOL_POST),
                                                   grad=PS.grad_ratio(g[:, sel], c["g_ref"][:, p])))
            else:
                for a, b in zip(base, (mu, var, dmu, dvar, val, g)):
                    assert _same(a, b), (M, path, unfused)


# ---- 2. every padded width -----------------------------------------------------------------------------------------

@pytest.mark.parametrize("n", [769, 2047])
@pytest.mark.parametrize("d", [1, 3, 5, 8, 10, 13, 20])
@pytest.mark.parametrize("kernel", [OB.KERNEL_MATERN52, KERNEL_MATERN12], ids=["matern52", "matern12"])
def test_every_padded_width(lib, kernel, d, n, monkeypatch):
    """Value and gradient calls whose default dispatch runs both the quarter path and the wide fused one: M = 300 and
    37888 without gradients, 37889 (a full chunk and a one-candidate tail) with them."""
    _env(monkeypatch, None, False)
    X, Y, ls, amp, ns = make_problem(n, d, seed=n * 31 + d)
    Xs = np.random.default_rng(d).random((d, 37889))
    Xs[:, 37888] = X[:, n - 1]                            # the tail candidate on the last training point
    sel = np.union1d(np.arange(300), _subset(37889, [PS.score_plan(n, 37889, d, True)], k=400))
    ref = Ref(kernel, X, Y[0], ls[0], amp[0], ns[0], Xs, sel)
    gp = lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], kid_of(lib, kernel))
    fam = f"width n={n}"
    for M in (300, 37888):
        mu, var, _ = lib.gp_predict(gp, Xs[:, :M])
        plan = _expect_paths(lib, n, M, d, False)
        assert [q["path"] for q in plan["passes"]] == (["quarter"] if M == 300 else ["wide_fused"])
        ref.check(f"{fam} value", sel[sel < M], mu, var)
    mu, var, dmu, dvar, _ = lib.gp_predict_grad([gp], 1, 1, Xs)
    plan = _expect_paths(lib, n, 37889, d, True, pgrad=True)
    assert [q["path"] for q in plan["passes"]] == ["wide_fused", "quarter"]
    ref.check(f"{fam} gradient", sel, mu[0], var[0], dmu[0], dvar[0])
    gp.free()


# ---- 3. batch-size edges -------------------------------------------------------------------------------------------

EDGE_M = [1, 31, 33, 8191, 8192, 8193, 37888, 37889, 75776 + 300, 75776 + 5000]


@pytest.fixture(scope="module")
def edge_problem(lib):
    n, d = 2048, 8
    X, Y, ls, amp, ns = make_problem(n, d, seed=4242)
    Xs = np.random.default_rng(4243).random((d, max(EDGE_M)))
    subs = {M: _subset(M, [PS.score_plan(n, M, d, False), PS.score_plan(n, M, d, True)], k=300) for M in EDGE_M}
    ref = Ref(OB.KERNEL_MATERN52, X, Y[0], ls[0], amp[0], ns[0], Xs, np.unique(np.concatenate(list(subs.values()))))
    gp = lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], OB.KERNEL_MATERN52)
    yield dict(n=n, d=d, Xs=Xs, subs=subs, ref=ref, gp=gp)
    gp.free()


def _alone_bits(lib, gp, Xs, edges, mu, var, dmu=None, dvar=None):
    """The chunk-boundary candidates scored one at a time give the same bits."""
    for m in edges:
        if dmu is None:
            a_mu, a_var, _ = lib.gp_predict(gp, Xs[:, m:m + 1])
        else:
            a_mu, a_var, a_dmu, a_dvar, _ = lib.gp_predict_grad([gp], 1, 1, Xs[:, m:m + 1])
            assert _same(a_dmu[0, :, 0], dmu[:, m]) and _same(a_dvar[0, :, 0], dvar[:, m]), m
        assert _same(np.ravel(a_mu)[:1], mu[m:m + 1]) and _same(np.ravel(a_var)[:1], var[m:m + 1]), m


@pytest.mark.parametrize("M", EDGE_M)
def test_batch_size_edges(lib, edge_problem, M, monkeypatch):
    _env(monkeypatch, None, False)
    c = edge_problem
    n, d, gp, ref, Xm, sel = c["n"], c["d"], c["gp"], c["ref"], c["Xs"][:, :M], c["subs"][M]
    mu, var, st = lib.gp_predict(gp, Xm)
    plan = _expect_paths(lib, n, M, d, False)
    ref.check("edges value", sel, mu, var)
    _alone_bits(lib, gp, Xm, PS.chunk_edges(plan, M), mu, var)
    mu_g, var_g, dmu, dvar, _ = lib.gp_predict_grad([gp], 1, 1, Xm)
    plan = _expect_paths(lib, n, M, d, True, pgrad=True)
    ref.check("edges gradient", sel, mu_g[0], var_g[0], dmu[0], dvar[0])
    assert _same(mu_g[0], mu) and _same(var_g[0], var)
    _alone_bits(lib, gp, Xm, PS.chunk_edges(plan, M), mu_g[0], var_g[0], dmu[0], dvar[0])


def test_narrow_tail_at_n4096(lib, monkeypatch):
    """M = 75777 at n = 4096: the last candidate is a chunk of its own and goes through the narrow kernel, 32 splits,
    with the chunk's leading dimension 75776 times its length."""
    _env(monkeypatch, None, False)
    n, d, M = 4096, 4, 75777
    X, Y, ls, amp, ns = make_problem(n, d, seed=4096)
    Xs = np.random.default_rng(4097).random((d, M))
    Xs[:, M - 1] = X[:, n - 1]
    plan = PS.score_plan(n, M, d, False)
    assert [(q["path"], q["nsp32"]) for q in plan["passes"]][1] == ("narrow", 32)
    sel = _subset(M, [plan, PS.score_plan(n, M, d, True)], k=300)
    ref = Ref(OB.KERNEL_MATERN52, X, Y[0], ls[0], amp[0], ns[0], Xs, sel)
    gp = lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], OB.KERNEL_MATERN52)
    mu, var, _ = lib.gp_predict(gp, Xs)
    _expect_paths(lib, n, M, d, False)
    ref.check("n=4096 tail value", sel, mu, var)
    _alone_bits(lib, gp, Xs, PS.chunk_edges(plan, M), mu, var)
    mu, var, dmu, dvar, _ = lib.gp_predict_grad([gp], 1, 1, Xs)
    gplan = _expect_paths(lib, n, M, d, True, pgrad=True)
    ref.check("n=4096 tail gradient", sel, mu[0], var[0], dmu[0], dvar[0])
    _alone_bits(lib, gp, Xs, PS.chunk_edges(gplan, M), mu[0], var[0], dmu[0], dvar[0])
    gp.free()


# ---- 4. Bayesian-inference samples x outputs -----------------------------------------------------------------------

def test_bi_samples_and_outputs(lib, monkeypatch):
    """y_dim = 3 outputs (Matern-5/2, Matern-1/2, RQ(3)) x S = 4 samples at n = 2048: every posterior of
    gp_predict_grad and the EI x PoF value and gradient with y_max, a box, a constraint mask and a prior mean with its
    gradient."""
    _env(monkeypatch, None, False)
    n, d, y_dim, S, M = 2048, 5, 3, 4, 3000
    kernels = [OB.KERNEL_MATERN52, KERNEL_MATERN12, RQ(3.0)]
    X, Y, ls, amp, ns = make_problem(n, d, seed=77, y_dim=y_dim)
    rng = np.random.default_rng(78)
    Xs = rng.random((d, M)) * 1.1 - 0.05                  # a few candidates outside the box
    Xs[:, 7] = X[:, 100]
    pm = 0.1 * rng.standard_normal((y_dim, M))
    pmg = 0.1 * rng.standard_normal((y_dim, d, M))
    gps, posts = [], []
    for s in range(S):
        row = []
        for i in range(y_dim):
            lss = ls[i] * (1 + 0.15 * s)
            gps.append(lib.gp_fit(X, Y[i], lss, amp[i], ns[i], kid_of(lib, kernels[i])))
            row.append(OK.posterior_fit(X, Y[i], lss, amp[i], ns[i], kernels[i]))
        posts.append(row)
    mu, var, dmu, dvar, st = lib.gp_predict_grad(gps, y_dim, S, Xs, pm, pmg)
    _expect_paths(lib, n, M, d, True, pgrad=True, nsl=y_dim * S)
    for s in range(S):
        for i in range(y_dim):
            q = s * y_dim + i
            rm, rv, rdm, rdv, rst = OK.mean_var_grad(posts[s][i], Xs, pm[i], pmg[i])
            lsq = ls[i] * (1 + 0.15 * s)
            b = PS.post_bounds(X, Y[i], lsq, amp[i], ns[i], kernels[i], Xs)
            _note("BI predict_grad", dict(mu=PS.ratio(mu[q], rm, PS.TOL_POST, b[0]), var=PS.ratio(var[q], rv, PS.TOL_POST, b[1]),
                                          dmu=PS.grad_ratio(dmu[q], rdm), dvar=PS.grad_ratio(dvar[q], rdv)))
    coefs, best = [1.0, 0.0, 0.0], float(np.quantile(Y[0], 0.8))
    y_max = [np.inf, float(np.quantile(Y[1], 0.7)), float(np.quantile(Y[2], 0.9))]
    lb, ub = np.zeros(d), np.ones(d)
    cm = (np.arange(M) % 11 != 3).astype(np.uint8)
    val, g = lib.ei_value_grad(gps, y_dim, S, Xs, coefs, best, y_max, lb, ub, cm, pm, pmg)
    _expect_paths(lib, n, M, d, True, nsl=y_dim * S)
    acq_ref = OK.ei_acquisition(posts, Xs, coefs, best, y_max, lb, ub, cm, pm)[0]
    g_ref = np.mean([OK.ei_value_grad(posts[s], Xs, coefs, best, y_max, pm, pmg)[1] for s in range(S)], axis=0)
    live = OB.in_bounds(Xs, lb, ub) & (cm != 0)
    g_ref = np.where(live[None], g_ref, 0.0)
    assert np.all(g[:, ~live] == 0.0) and np.all(val[~live] == 0.0)
    _note("BI ei_value_grad", dict(val=PS.grad_ratio(val[None], acq_ref[None], PS.TOL_POST), grad=PS.grad_ratio(g, g_ref)))
    acq, _, _ = lib.ei_score(gps, y_dim, S, Xs, coefs, best, y_max, lb, ub, cm, pm)
    assert _same(acq, val)
    for gp in gps:
        gp.free()


def test_predict_grad_across_pgrad_slots(lib, monkeypatch):
    """y_dim = 8, S = 2, d = 32: the output slot caps the chunk at 246 candidate blocks; M = 31 688 runs two chunks."""
    _env(monkeypatch, None, False)
    n, d, y_dim, S = 300, 32, 8, 2
    M = 246 * 128 + 200
    X, Y, ls, amp, ns = make_problem(n, d, seed=88, y_dim=y_dim)
    Xs = np.random.default_rng(89).random((d, M))
    gps, refs = [], []
    plan = PS.score_plan(n, M, d, True, pgrad=True, nsl=y_dim * S)
    assert plan["CH"] == 246 * 128
    sel = _subset(M, [plan], k=200)
    for s in range(S):
        for i in range(y_dim):
            lss = ls[i] * (1 + 0.3 * s)
            gps.append(lib.gp_fit(X, Y[i], lss, amp[i], ns[i], OB.KERNEL_MATERN52))
            refs.append(Ref(OB.KERNEL_MATERN52, X, Y[i], lss, amp[i], ns[i], Xs, sel))
    mu, var, dmu, dvar, st = lib.gp_predict_grad(gps, y_dim, S, Xs)
    _expect_paths(lib, n, M, d, True, pgrad=True, nsl=y_dim * S)
    for q, r in enumerate(refs):
        r.check("PGRAD slots", sel, mu[q], var[q], dmu[q], dvar[q])
    for gp in gps:
        gp.free()


# ---- 5. slices of different block counts in one call ---------------------------------------------------------------

@pytest.mark.parametrize("n0", [128, 2048])
def test_mixed_slices(lib, n0, monkeypatch):
    """Two outputs whose GPs have n0 and n0 + 1 points (the second grown by boss_gp_append at n0 = 2048): the slices
    take different paths or block counts, and the chunk buffers are sized by the larger."""
    _env(monkeypatch, None, False)
    d = 4
    X, Y, ls, amp, ns = make_problem(n0 + 1, d, seed=n0 + 5, y_dim=2)
    g0 = lib.gp_fit(X[:, :n0], Y[0, :n0], ls[0], amp[0], ns[0], OB.KERNEL_MATERN52)
    if n0 == 2048:
        g1 = lib.gp_fit(X[:, :n0], Y[1, :n0], ls[1], amp[1], ns[1], OB.KERNEL_MATERN52)
        assert lib.gp_append(g1, X[:, n0], Y[1, n0])
    else:
        g1 = lib.gp_fit(X, Y[1], ls[1], amp[1], ns[1], OB.KERNEL_MATERN52)
    ns_ = [n0, n0 + 1]
    best = float(np.quantile(Y[0], 0.9))
    y_max = [np.inf, float(np.quantile(Y[1], 0.8))]
    for M in (40, 3000, 37888):
        Xs = np.random.default_rng(M).random((d, M))
        sel = _subset(M, [PS.score_plan(ns_, M, d, True)], k=300)
        refs = [Ref(OB.KERNEL_MATERN52, X[:, :n0], Y[0, :n0], ls[0], amp[0], ns[0], Xs, sel),
                Ref(OB.KERNEL_MATERN52, X, Y[1], ls[1], amp[1], ns[1], Xs, sel)]
        mu, var, dmu, dvar, _ = lib.gp_predict_grad([g0, g1], 2, 1, Xs)
        plan = _expect_paths(lib, ns_, M, d, True, pgrad=True)
        if n0 == 128:
            assert {p["path"] for p in plan["passes"] if p["slice"] == 0} != {p["path"] for p in plan["passes"] if p["slice"] == 1}
        for q in range(2):
            refs[q].check(f"mixed slices n={n0}", sel, mu[q], var[q], dmu[q], dvar[q])
        val, g = lib.ei_value_grad([g0, g1], 2, 1, Xs, [1.0, 0.0], best, y_max)
        _expect_paths(lib, ns_, M, d, True)
        posts = [[refs[0].post, refs[1].post]]
        acq_ref = OB.ei_acquisition(posts, Xs[:, sel], [1.0, 0.0], best, y_max)[0]
        g_ref = OB.ei_value_grad(posts[0], Xs[:, sel], [1.0, 0.0], best, y_max)[1]
        _note(f"mixed slices n={n0} ei", dict(val=PS.grad_ratio(val[sel][None], acq_ref[None], PS.TOL_POST),
                                             grad=PS.grad_ratio(g[:, sel], g_ref)))
        acq, _, _ = lib.ei_score([g0, g1], 2, 1, Xs, [1.0, 0.0], best, y_max)
        _expect_paths(lib, ns_, M, d, False)
        assert _same(acq, val)
    # argmax only: screened and unscreened calls give the same pair
    M = 20000
    Xs = np.random.default_rng(7).random((d, M))
    monkeypatch.setenv("BOSS_SCREEN_MIN_M", "1")
    _, bv, bi = lib.ei_score([g0, g1], 2, 1, Xs, [1.0, 0.0], best, y_max, want_acq=False)
    assert lib.dbg_screen_stats()[0] != 0                 # the screen ran (possibly falling back after chunk 1)
    monkeypatch.setenv("BOSS_NO_SCREEN", "1")
    _, bv2, bi2 = lib.ei_score([g0, g1], 2, 1, Xs, [1.0, 0.0], best, y_max, want_acq=False)
    assert lib.dbg_screen_stats()[0] == 0
    _expect_paths(lib, ns_, M, d, False)
    assert bi == bi2 and _same([bv], [bv2])
    acq, bv3, bi3 = lib.ei_score([g0, g1], 2, 1, Xs, [1.0, 0.0], best, y_max)
    assert bi3 == bi and bi == OB.julia_argmax_fast(acq)
    g0.free()
    g1.free()


# ---- 6. boss_gp_append at scale ------------------------------------------------------------------------------------

def _check_factors(family, lib, gp, X, y, ls, amp, ns, kernel):
    """L, W = L^-1, alpha and the log-likelihood of a handle against the FP64 refit; -> the reference posterior."""
    Om = PS.reference(kernel)
    post = Om.posterior_fit(X, y, ls, amp, ns, kernel)
    L, W, al = lib.dbg_factors(gp)
    Lref = post.U.T
    Wref = sl.solve_triangular(Lref, np.eye(Lref.shape[0]), lower=True, check_finite=False)
    _note(family, dict(L=np.max(np.abs(L - Lref)) / (1e-10 * np.max(np.abs(Lref))),
                       W=np.max(np.abs(W - Wref)) / (1e-9 * np.max(np.abs(Wref))),
                       alpha=np.max(np.abs(al - post.alpha_w)) / (1e-9 * np.max(np.abs(post.alpha_w))),
                       loglik=abs(gp.loglik - Om.gp_loglik(X, y, ls, amp, ns, kernel)) / (1e-8 * abs(gp.loglik))))
    return post


def _cov_check(family, lib, gp, post, Xs):
    mu, cov, rc = lib.gp_cov(gp, Xs)
    Om = PS.reference(post.kernel_id)
    C_ref, st = Om.posterior_cov(post, Xs)
    mu_ref = Om.mean_and_var(post, Xs)[0]
    assert rc == 0 and not st.any()
    scale = np.sqrt(np.outer(np.diag(C_ref), np.diag(C_ref)))
    _note(family, dict(cov_mu=relerr(mu, mu_ref) / PS.TOL_POST, cov=float(np.max(np.abs(cov - C_ref) / scale)) / PS.TOL_POST))
    assert np.array_equal(cov, cov.T)


APPEND_CASES = [(k, 2040, 20) for k in KERNELS] + [(OB.KERNEL_MATERN52, 4090, 10)]


@pytest.mark.parametrize("kernel,n0,m", APPEND_CASES, ids=[f"{i}-{n0}+{m}" for i, (_, n0, m) in
                                                           zip(IDS + ["matern52"], APPEND_CASES)])
def test_append_at_scale(lib, kernel, n0, m, monkeypatch):
    """Fit n0 points and append m one at a time, across the 2048 -> 2049 (16 -> 17 blocks) or 4096 -> 4097 capacity
    repack; factors, log-likelihood, posterior, gradients and covariance of the grown handle against a refit."""
    _env(monkeypatch, None, False)
    n, d = n0 + m, 4
    X, Y, ls, amp, ns = make_problem(n, d, seed=n0 + m)
    gp = lib.gp_fit(X[:, :n0], Y[0, :n0], ls[0], amp[0], ns[0], kid_of(lib, kernel))
    for k in range(n0, n):
        assert lib.gp_append(gp, X[:, k], Y[0, k])
    assert gp.n == n
    post = _check_factors(f"append n={n0}+{m}", lib, gp, X, Y[0], ls[0], amp[0], ns[0], kernel)
    Xs = np.random.default_rng(n).random((d, 600))
    Xs[:, 0] = X[:, n - 1]                                # on the last appended point
    ref = Ref(kernel, X, Y[0], ls[0], amp[0], ns[0], Xs, np.arange(600))
    for path in ("quarter", "wide"):
        _env(monkeypatch, path, False)
        mu, var, dmu, dvar, _ = lib.gp_predict_grad([gp], 1, 1, Xs)
        _expect_paths(lib, n, 600, d, True, pgrad=True, path=path)
        ref.check(f"append n={n0}+{m} {path}", np.arange(600), mu[0], var[0], dmu[0], dvar[0])
    _env(monkeypatch, None, False)
    _cov_check(f"append n={n0}+{m}", lib, gp, post, Xs[:, :256])
    gp.free()


# ---- 7. single fit and covariance ----------------------------------------------------------------------------------

@pytest.mark.parametrize("n", [2048, 4096])
@pytest.mark.parametrize("kernel", [KERNEL_MATERN12, RQ(0.5), RQ(3.0)], ids=["matern12", "rq0.5", "rq3"])
def test_single_fit_and_cov(lib, kernel, n):
    d = 6
    X, Y, ls, amp, ns = make_problem(n, d, seed=n + 13)
    gp = lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], kid_of(lib, kernel))
    post = _check_factors(f"fit n={n}", lib, gp, X, Y[0], ls[0], amp[0], ns[0], kernel)
    _cov_check(f"cov n={n}", lib, gp, post, np.random.default_rng(n).random((d, 256)))
    gp.free()


@pytest.mark.parametrize("kernel", KERNELS, ids=IDS)
def test_cov_every_kernel(lib, kernel):
    n, d = 2048, 5
    X, Y, ls, amp, ns = make_problem(n, d, seed=5150)
    gp = lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], kid_of(lib, kernel))
    post = PS.reference(kernel).posterior_fit(X, Y[0], ls[0], amp[0], ns[0], kernel)
    Xs = np.random.default_rng(5151).random((d, 256))
    Xs[:, 3] = X[:, 9]
    _cov_check("cov n=2048 M=256", lib, gp, post, Xs)
    gp.free()
