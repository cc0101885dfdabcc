"""Device top-k of the closed-form EI (boss_ei_score_topk, DESIGN.md 2.10).  The k best (value, index) pairs must be,
bit for bit, the first k of the full score vector ordered by Julia's stable sortperm(vals; rev=true): descending under
isless (NaN first, all NaNs equal, +0.0 before -0.0), ties to the lower index.  The order reference below and its key
transform are tested without a GPU; the GPU cases compare the device selection, screened and unscreened, against it."""
import numpy as np
import pytest

from tests.util_problems import make_problem

gpu = pytest.mark.gpu
M = 200_000   # several 75 776-candidate chunks at n <= 4096: the running set and the screening pool span chunks
KS = [1, 7, 128, 1000, 8192]
# The bound separates the k best from the rest only while the k-th best score stays far above the typical bound: at
# the bench shape k <= 7 screens with a small pool, and from k ~ 100 on more than a quarter of the first chunk
# survives and the call falls back (results are compared in every state).


# ---- host reference of the order ----------------------------------------------------------------------------------

def isless_key(v):
    """uint64 keys whose unsigned order is Julia's isless: NaN the top key, negative -> ~bits, else bits | 1 << 63."""
    v = np.asarray(v, dtype=np.float64)
    u = np.ascontiguousarray(v).view(np.uint64)
    k = np.where((u >> np.uint64(63)) != 0, ~u, u | np.uint64(1 << 63))
    return np.where(np.isnan(v), np.uint64(0xFFFFFFFFFFFFFFFF), k)


def ref_order(v):
    """Stable descending sort under isless, written without the key: NaN first, then value descending, +0.0 before
    -0.0, then index ascending."""
    v = np.asarray(v, dtype=np.float64)
    nan = np.isnan(v)
    vv = np.where(nan, 0.0, v)
    return np.lexsort((np.arange(v.size), np.signbit(vv), -vv, ~nan))


def _bits(v):
    return np.ascontiguousarray(np.asarray(v, dtype=np.float64)).view(np.int64)


SPECIAL = np.array([0.0, -0.0, np.inf, -np.inf, np.nan, 5e-324, -5e-324, 2.2250738585072014e-308, 1.0, -1.0, 1.0, 0.0,
                    -0.0, np.nan, -np.nan, np.finfo(np.float64).max, -np.finfo(np.float64).max, 1e-300, -1e-300])


def test_isless_key_orders_special_values():
    k = isless_key(SPECIAL)
    assert k[4] == k[13] == k[14] == np.uint64(0xFFFFFFFFFFFFFFFF)          # every NaN is the top key, sign ignored
    assert k[1] < k[0] and k[6] < k[1] and k[0] < k[5] < k[7]                # -tiny < -0.0 < +0.0 < subnormal < normal
    assert k[3] < k[16] < k[9] < k[6] and k[8] < k[15] < k[2] < k[4]          # -Inf lowest, +Inf below NaN
    assert k[8] == k[10] and k[0] == k[11] and k[1] == k[12]                  # equal values, equal keys
    finite = ~np.isnan(SPECIAL)
    f = SPECIAL[finite]
    kf = k[finite]
    for i in range(f.size):                                                  # key order == value order, -0.0 < +0.0
        for j in range(f.size):
            lt = f[i] < f[j] or (f[i] == f[j] == 0.0 and np.signbit(f[i]) and not np.signbit(f[j]))
            assert (kf[i] < kf[j]) == lt, (f[i], f[j])


def test_reference_order_matches_key_order_and_ties():
    rng = np.random.default_rng(3)
    v = np.concatenate([SPECIAL, rng.choice(SPECIAL, 500), rng.standard_normal(300), np.zeros(50)])
    rng.shuffle(v)
    o = ref_order(v)
    assert np.array_equal(o, np.argsort(~isless_key(v), kind="stable"))
    k = isless_key(v)[o]
    assert np.all(k[:-1] >= k[1:])
    same = k[:-1] == k[1:]
    assert np.all(o[:-1][same] < o[1:][same])                                 # ties: ascending index
    assert np.isnan(v[o[0]]) and o[0] == np.flatnonzero(np.isnan(v))[0]
    # without NaN, the old mirror order (np.argsort(-vals, kind="stable")) is the same up to the sign of zero
    w = np.where(np.isnan(v), 1.0, v)
    w[w == 0.0] = 0.0
    assert np.array_equal(ref_order(w), np.argsort(-w, kind="stable"))


def test_mirror_sortperm_and_argmax_agree_with_reference():
    from boss_b200.acquisition import julia_argmax, julia_sortperm_rev
    rng = np.random.default_rng(4)
    for _ in range(20):
        v = rng.choice(SPECIAL, 200)
        assert np.array_equal(julia_sortperm_rev(v), ref_order(v))
        assert julia_sortperm_rev(v)[0] == julia_argmax(v)


# ---- device ------------------------------------------------------------------------------------------------------

def _check(tv, ti, acq, k):
    o = ref_order(acq)[:k]
    assert tv.shape == (k,) and ti.shape == (k,)
    assert np.array_equal(ti, o), (ti[:8], o[:8])
    assert np.array_equal(_bits(tv), _bits(acq[o]))


def _ref_scores(lib, monkeypatch, *args, **kw):
    monkeypatch.setenv("BOSS_NO_SCREEN", "1")
    acq, bv, bi = lib.ei_score(*args, want_acq=True, **kw)
    monkeypatch.delenv("BOSS_NO_SCREEN")
    return acq, bv, bi


def _both(lib, monkeypatch, call, acq, k):
    """call() screened (BOSS_SCREEN_MIN_M=4096) and with BOSS_NO_SCREEN=1; both must equal the reference.  Returns the
    screened call's counters."""
    monkeypatch.setenv("BOSS_SCREEN_MIN_M", "4096")
    monkeypatch.delenv("BOSS_NO_SCREEN", raising=False)
    tv, ti = call()
    st = lib.dbg_screen_stats()
    _check(tv, ti, acq, k)
    monkeypatch.setenv("BOSS_NO_SCREEN", "1")
    tv, ti = call()
    assert lib.dbg_screen_stats()[0] == 0
    _check(tv, ti, acq, k)
    monkeypatch.delenv("BOSS_NO_SCREEN")
    return st


def _fit(lib, n, d, seed, y_dim=1):
    X, Y, ls, amp, ns = make_problem(n, d, seed=seed, y_dim=y_dim)
    gps = [lib.gp_fit(X, Y[i], ls[i], amp[i], ns[i], lib.KERNEL_MATERN52) for i in range(y_dim)]
    return X, Y, gps


@pytest.fixture(scope="module")
def bench(lib):
    """bench.py's shape: n = 2048, d = 8, with the full score vector of the unscreened path."""
    import os
    X, Y, gps = _fit(lib, 2048, 8, 1002)
    Xs = np.random.default_rng(7).random((8, M))
    best = float(np.max(Y[0]))
    os.environ["BOSS_NO_SCREEN"] = "1"
    try:
        acq, bv, bi = lib.ei_score(gps, 1, 1, Xs, [1.0], best, None, want_acq=True)
    finally:
        del os.environ["BOSS_NO_SCREEN"]
    yield gps[0], best, Xs, acq, (bv, bi)
    gps[0].free()


@gpu
@pytest.mark.parametrize("k", KS)
def test_bench_shape(lib, monkeypatch, bench, k):
    gp, best, Xs, acq, _ = bench
    st = _both(lib, monkeypatch, lambda: lib.ei_score_topk([gp], 1, 1, Xs, [1.0], best, None, k), acq, k)
    if k <= 7:
        assert st[0] == 1 and st[1] == M and k <= st[2] < M // 10, st
    else:
        assert st[0] in (1, 2), st


@gpu
def test_top1_is_the_argmax_pair(lib, monkeypatch, bench):
    gp, best, Xs, acq, (bv0, bi0) = bench
    monkeypatch.delenv("BOSS_NO_SCREEN", raising=False)
    _, bv, bi = lib.ei_score([gp], 1, 1, Xs, [1.0], best, None, want_acq=False)     # screened argmax
    assert lib.dbg_screen_stats()[0] == 1
    for k in (1, 64):
        tv, ti = lib.ei_score_topk([gp], 1, 1, Xs, [1.0], best, None, k)
        assert (int(_bits(tv[0])), int(ti[0])) == (int(_bits(bv)), bi) == (int(_bits(bv0)), bi0)


@gpu
def test_host_pinned_and_device_inputs(lib, monkeypatch, bench):
    import torch
    gp, best, Xs, acq, _ = bench
    pinned = torch.empty((M, 8), dtype=torch.float64, pin_memory=True)
    pinned.copy_(torch.from_numpy(np.ascontiguousarray(Xs.T)))
    dev = pinned.cuda()
    torch.cuda.synchronize()
    for k in (7, 128):
        st = _both(lib, monkeypatch, lambda: lib.ei_score_topk([gp], 1, 1, pinned.numpy().T, [1.0], best, None, k), acq, k)
        assert st[0] == (1 if k == 7 else 2), st
        st = _both(lib, monkeypatch, lambda: lib.ei_score_topk_dev([gp], 1, 1, dev.data_ptr(), M, [1.0], best, None, k),
                   acq, k)
        assert st[0] == (1 if k == 7 else 2), st


@gpu
def test_bi_samples(lib, monkeypatch):
    n, d = 512, 5
    X, Y, ls, amp, ns = make_problem(n, d, seed=41)
    gps = [lib.gp_fit(X, Y[0], ls[0] * f, amp[0] * g, ns[0], lib.KERNEL_MATERN52)
           for f, g in ((1.0, 1.0), (0.8, 1.2), (1.3, 0.9))]
    Xs = np.random.default_rng(42).random((d, M))
    best = float(np.max(Y[0]))
    acq, _, _ = _ref_scores(lib, monkeypatch, gps, 1, 3, Xs, [1.0], best, None)
    for k in (5, 300):
        st = _both(lib, monkeypatch, lambda: lib.ei_score_topk(gps, 1, 3, Xs, [1.0], best, None, k), acq, k)
        assert st[0] in (1, 2), st


@gpu
def test_two_outputs_coefs_ymax_bounds_mask_prior_mean_and_no_best(lib, monkeypatch):
    n, d = 2048, 8
    X, Y, gps = _fit(lib, n, d, 43, y_dim=2)
    rng = np.random.default_rng(44)
    Xs = rng.random((d, M)) * 1.2 - 0.1            # some candidates outside [0, 1]^d
    coefs = np.array([1.0, -0.5])
    y_max = np.array([np.inf, float(np.quantile(Y[1], 0.8))])
    best = float(np.max(coefs @ Y))
    cm = (rng.random(M) > 0.2).astype(np.uint8)
    pm = 0.05 * rng.standard_normal((2, M))
    lb, ub = np.zeros(d), np.ones(d)
    k = 5
    cases = [dict(y_max=y_max), dict(y_max=y_max, lb=lb, ub=ub, cons_mask=cm, prior_mean_s=pm),
             dict(y_max=None, lb=lb, ub=ub, cons_mask=cm), dict(y_max=None, lb=lb, ub=ub, cons_mask=cm, prior_mean_s=pm)]
    for kw in cases:
        ym = kw.pop("y_max")
        acq, _, _ = _ref_scores(lib, monkeypatch, gps, 2, 1, Xs, coefs, best, ym, **kw)
        st = _both(lib, monkeypatch, lambda: lib.ei_score_topk(gps, 2, 1, Xs, coefs, best, ym, k, **kw), acq, k)
        assert st[0] in (1, 2), st
    # best = None (no feasible observation): scores are PoF only, never screened
    acq, _, _ = _ref_scores(lib, monkeypatch, gps, 2, 1, Xs, coefs, None, y_max, lb=lb, ub=ub)
    st = _both(lib, monkeypatch, lambda: lib.ei_score_topk(gps, 2, 1, Xs, coefs, None, y_max, 1000, lb=lb, ub=ub), acq, 1000)
    assert st[0] == 0, st


@gpu
def test_duplicated_candidates_tie_to_the_lower_index(lib, monkeypatch, bench):
    gp, best, Xs, _, _ = bench
    Xd = np.repeat(Xs[:, : M // 4], 4, axis=1)     # every candidate four times in a row
    acq, _, _ = _ref_scores(lib, monkeypatch, [gp], 1, 1, Xd, [1.0], best, None)
    for k in (7, 1000):
        st = _both(lib, monkeypatch, lambda: lib.ei_score_topk([gp], 1, 1, Xd, [1.0], best, None, k), acq, k)
        assert st[0] == (1 if k == 7 else 2), st


@gpu
def test_zeros_across_the_kth_boundary_fall_back(lib, monkeypatch, bench):
    """Only 500 candidates lie inside the bounds: the 1000-th best score is 0, the seed's T is 0 and the call falls
    back to the full path, whose running set then ends in a long run of tied zeros (lowest indices kept)."""
    gp, best, Xs, _, _ = bench
    Xz = Xs.copy()
    out = np.ones(M, dtype=bool)
    out[np.random.default_rng(9).choice(M, 500, replace=False)] = False
    Xz[0, out] += 2.0
    lb, ub = np.zeros(8), np.ones(8)
    acq, _, _ = _ref_scores(lib, monkeypatch, [gp], 1, 1, Xz, [1.0], best, None, lb=lb, ub=ub)
    for k in (499, 1000, 8192):
        st = _both(lib, monkeypatch, lambda: lib.ei_score_topk([gp], 1, 1, Xz, [1.0], best, None, k, lb=lb, ub=ub), acq, k)
        if k > 500:
            assert st[0] == 2, st


@gpu
def test_nan_and_failed_variance_candidates(lib, monkeypatch, bench):
    """A NaN prior mean makes the score NaN (ranked first, all NaNs equal, ties to the lower index); a NaN coordinate
    fails _clip_var and scores -Inf (ranked last)."""
    gp, best, Xs, _, _ = bench
    Xn = Xs.copy()
    Xn[1, [150_001, 90_000, 150_000, 7]] = np.nan
    pm = np.zeros((1, M))
    pm[0, [180_000, 3, 120_000]] = np.nan
    acq, _, _ = _ref_scores(lib, monkeypatch, [gp], 1, 1, Xn, [1.0], best, None, prior_mean_s=pm)
    assert np.isnan(acq).sum() == 3 and np.isneginf(acq).sum() == 4
    for k in (2, 3, 200):
        st = _both(lib, monkeypatch, lambda: lib.ei_score_topk([gp], 1, 1, Xn, [1.0], best, None, k, prior_mean_s=pm),
                   acq, k)
        assert st[0] in (1, 2), st
    # -Inf entries inside the selection: k = M of a small batch reaches them
    m = 5000
    acq_s, _, _ = _ref_scores(lib, monkeypatch, [gp], 1, 1, Xn[:, :m], [1.0], best, None, prior_mean_s=pm[:, :m])
    tv, ti = lib.ei_score_topk([gp], 1, 1, Xn[:, :m], [1.0], best, None, m, prior_mean_s=pm[:, :m])
    _check(tv, ti, acq_s, m)
    assert np.isneginf(tv[-1]) and np.isnan(tv[0])


@gpu
def test_k_equal_m_and_out_of_range(lib, monkeypatch, bench):
    gp, best, Xs, acq, _ = bench
    m = 8192
    acq_s, _, _ = _ref_scores(lib, monkeypatch, [gp], 1, 1, Xs[:, :m], [1.0], best, None)
    tv, ti = lib.ei_score_topk([gp], 1, 1, Xs[:, :m], [1.0], best, None, m)
    _check(tv, ti, acq_s, m)
    assert sorted(ti.tolist()) == list(range(m))
    tv, ti = lib.ei_score_topk([gp], 1, 1, Xs[:, :1], [1.0], best, None, 1)
    _check(tv, ti, acq[:1], 1)
    for k in (0, -1, 11, 8193):
        with pytest.raises(lib.BossError):
            lib.ei_score_topk([gp], 1, 1, Xs[:, :10] if k == 11 else Xs[:, :9000], [1.0], best, None, k)
    assert lib.lib.boss_ei_score_topk(None, 1, 1, None, 0, None, None, None, None, None, None, None, 1, None, None) == -1


@gpu
def test_sample_opt_am_starts_match_the_host_sort(lib):
    """maximize_acquisition(SampleOptAM) takes its starts from Acquisition.topk; on a NaN-free problem they are the
    ones the old host path picked: every score to the host, then np.argsort(-vals, kind="stable")[:multistart]."""
    import boss_b200 as B
    from boss_b200 import acquisition_maximizers as AMs
    rng = np.random.default_rng(0)
    f = lambda x: np.array([np.sin(x[0]) + 0.5 * np.cos(2 * x[1])])
    dom = B.Domain(([0.0, 0.0], [10.0, 10.0]))
    X = B.generate_LHC(dom.bounds, 20, rng)
    Y = np.stack([f(X[:, j]) for j in range(20)], axis=1)
    model = B.GaussianProcess(kernel=B.SqExponentialKernel(),
                              lengthscale_priors=[B.mvlognormal([0.5, 0.5], [0.5, 0.5])],
                              amplitude_priors=[B.LogNormal(0.0, 0.5)], noise_std_priors=[B.Dirac(0.1)])
    prob = B.BossProblem(f, dom, B.ExpectedImprovement(B.LinFitness([1.0])), model, B.ExperimentData(X, Y))
    prob.params = B.estimate_parameters(B.SamplingMAP(64, seed=1), prob)
    acq = B.construct_acquisition(prob)
    am = B.SampleOptAM(None, 3000, 16, iters=20, seed=5)
    x_new, v_new = B.maximize_acquisition(am, prob, acq=acq)
    # the old path, restated: same sampler seed, all scores, host sort
    old = B.SampleOptAM(None, 3000, 16, iters=20, seed=5)
    Xo, vals = B.maximize_acquisition(old.sampler, prob, return_all=True, acq=acq)
    assert not np.isnan(vals).any()
    top_old = np.argsort(-vals, kind="stable")[:16]
    top_new, tv = acq.topk(Xo, 16)
    assert np.array_equal(top_new, top_old) and np.array_equal(_bits(tv), _bits(vals[top_old]))
    x_old, v_old = B.maximize_acquisition(AMs.OptimizationAM(Xo[:, top_old], old.iters), prob, acq=acq)
    assert np.array_equal(x_new, x_old) and int(_bits(v_new)) == int(_bits(v_old))


def _n_gpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


@gpu
@pytest.mark.skipif(_n_gpus() < 2, reason="needs >= 2 GPUs")
def test_multi_gpu_in_library_matches_single_gpu(lib, monkeypatch, bench):
    """Last in the module: the process keeps driving two devices afterwards."""
    gp, best, Xs, acq, _ = bench
    X, Y, ls, amp, ns = make_problem(2048, 8, seed=1002)
    lib.init_multi(2)
    assert lib.n_devices() == 2
    g2 = lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], lib.KERNEL_MATERN52)
    for screen in (True, False):
        if not screen:
            monkeypatch.setenv("BOSS_NO_SCREEN", "1")
        for k in (1, 1000, 8192):
            tv, ti = lib.ei_score_topk([g2], 1, 1, Xs, [1.0], best, None, k)
            _check(tv, ti, acq, k)
    g2.free()
