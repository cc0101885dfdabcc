"""The FP32 mean tier of argmax screening and the re-seeded threshold (DESIGN.md 2.9).

- The error bound holds: |mu~ - mu64| <= E for every candidate, over the three covariance functions, every padded
  input dimension, extreme length-scales, near-duplicate training points, tiny noise, discrete dimensions, candidates
  far outside the box and BI samples.
- The FP32 kappa stays within the evaluation budget of E over r in [0, 40].
- The pool is the FP64 tier's: with BOSS_SCREEN_NO_RESEED=1 the two tiers keep the same number of candidates, and the
  pairs / top-k lists equal the unscreened call's bit for bit.
- The re-seed is sound: with it on the results are unchanged and the pool is no larger.
"""
import numpy as np
import pytest

from tests.util_problems import make_problem

pytestmark = pytest.mark.gpu

M = 200_000   # several 75 776-candidate chunks at n <= 4096, so the FP32 tier takes part


def _bits(v):
    return int(np.array(v, dtype=np.float64).view(np.int64))


def _bound_ratio(lib, gp, Xs):
    mu32, E, mu64 = lib.dbg_screen_mean(gp, Xs)
    assert np.all(np.isfinite(E)) and np.all(E > 0)
    fin = np.isfinite(mu64)
    err = np.abs(mu32[fin] - mu64[fin])
    ratio = float(np.max(err / E[fin]))
    assert ratio <= 1.0, ratio
    return ratio


def _gp(lib, n, d, seed, kid, ls_scale=1.0, noise=0.1, dup=False, disc=None):
    X, Y, ls, amp, ns = make_problem(n, d, seed=seed, noise=noise)
    if dup:   # every other training point a near-duplicate of its neighbour
        X[:, 1::2] = X[:, 0::2][:, : X[:, 1::2].shape[1]] + 1e-9
    if disc is not None:
        X[disc] = np.round(4 * X[disc])
    gp = lib.gp_fit(X, Y[0], ls[0] * ls_scale, amp[0], ns[0], kid,
                    discrete_mask=None if disc is None else disc.astype(np.uint8))
    assert gp is not None
    return gp


KIDS = ("KERNEL_SE", "KERNEL_MATERN32", "KERNEL_MATERN52")


@pytest.mark.parametrize("kid", KIDS)
@pytest.mark.parametrize("d", [1, 2, 3, 4, 5, 6, 7, 8, 11, 12, 16, 17, 32])
def test_bound_holds_every_kernel_and_padded_dim(lib, kid, d):
    gp = _gp(lib, 700, d, 100 + d, getattr(lib, kid))
    Xs = np.random.default_rng(d).random((d, 20_000))
    _bound_ratio(lib, gp, Xs)
    gp.free()


def test_bound_holds_bench_problem(lib):
    X, Y, ls, amp, ns = make_problem(2048, 8, seed=1002)
    gp = lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], lib.KERNEL_MATERN52)
    ratio = _bound_ratio(lib, gp, np.random.default_rng(7).random((8, 65_536)))
    print(f"bench problem: max |mu~ - mu64| / E = {ratio:.3e}")
    gp.free()


@pytest.mark.parametrize("kid", KIDS)
@pytest.mark.parametrize("case", ["ls_small", "ls_large", "near_dup", "noise_1e-6", "discrete", "far_out"])
def test_bound_holds_hard_cases(lib, kid, case):
    d, n = 6, (200 if case == "noise_1e-6" else 1024)
    kw = {"ls_small": dict(ls_scale=1e-2), "ls_large": dict(ls_scale=1e2), "near_dup": dict(dup=True),
          "noise_1e-6": dict(noise=1e-6), "discrete": dict(disc=np.array([1, 0, 1, 0, 0, 0], dtype=bool)),
          "far_out": {}}[case]
    gp = _gp(lib, n, d, 7, getattr(lib, kid), **kw)
    rng = np.random.default_rng(8)
    Xs = rng.random((d, 20_000))
    if case == "far_out":
        Xs = Xs * 200.0 - 100.0
        Xs[:, :10] = 1e40          # beyond FP32: the rounded point is infinite, mu~ is 0 (SE) or NaN (Matern)
    if case == "discrete":
        Xs[[0, 2]] *= 4.0
    mu32, E, mu64 = lib.dbg_screen_mean(gp, Xs)
    fin = np.isfinite(mu32) & np.isfinite(mu64)
    assert np.all(np.abs(mu32[fin] - mu64[fin]) <= E[fin])
    gp.free()


def test_bound_holds_bi_samples(lib):
    X, Y, ls, amp, ns = make_problem(512, 5, seed=41)
    rng = np.random.default_rng(42).random((5, 20_000))
    for f, g in ((1.0, 1.0), (0.8, 1.2), (1.3, 0.9)):
        gp = lib.gp_fit(X, Y[0], ls[0] * f, amp[0] * g, ns[0], lib.KERNEL_MATERN52)
        _bound_ratio(lib, gp, rng)
        gp.free()


@pytest.mark.parametrize("kid", [0, 1, 2])
def test_kappa_f32_within_evaluation_budget(lib, kid):
    """|kappa~(r) - kappa(r)| over r in [0, 40], in units of 2^-24, at the FP32-rounded d2: the evaluation part of
    SCREEN_C_EVAL (64), which also carries the rounding of r and of the runs of 8."""
    r = np.concatenate([np.linspace(0.0, 40.0, 400_001), np.geomspace(1e-20, 1e-2, 2000)])
    d2 = (r * r).astype(np.float32).astype(np.float64)
    s = np.sqrt(d2)
    ref = [np.exp(-0.5 * d2), (1 + np.sqrt(3) * s) * np.exp(-np.sqrt(3) * s),
           (1 + np.sqrt(5) * s + 5 / 3 * d2) * np.exp(-np.sqrt(5) * s)][kid]
    got = lib.dbg_kappa_f32(kid, r)
    err = np.abs(got - ref)
    i = int(np.argmax(err))
    worst = float(err[i] / 2.0**-24)
    print(f"kid {kid}: max |kappa~ - kappa| = {worst:.2f} * 2^-24 at r = {r[i]:.6g}")
    assert worst <= 16.0, (worst, r[i], got[i], ref[i])


# ---- the pool and the results ----

def _run(lib, monkeypatch, call, env):
    for k in ("BOSS_NO_SCREEN", "BOSS_SCREEN_F64", "BOSS_SCREEN_NO_RESEED"):
        monkeypatch.delenv(k, raising=False)
    for k in env:
        monkeypatch.setenv(k, "1")
    out = call()
    return out, lib.dbg_screen_stats(), lib.dbg_screen_ambiguous()


def _tiers(lib, monkeypatch, call, key):
    """call() under the FP64 tier, the FP32 tier without and with re-seed, and unscreened: results equal bit for bit,
    the two tiers' pools equal in size, the re-seeded pool no larger.  Returns the FP32 tier's counters."""
    monkeypatch.setenv("BOSS_SCREEN_MIN_M", "4096")
    ref, st0, _ = _run(lib, monkeypatch, call, ["BOSS_NO_SCREEN"])
    assert st0[0] == 0
    r64, st64, _ = _run(lib, monkeypatch, call, ["BOSS_SCREEN_F64", "BOSS_SCREEN_NO_RESEED"])
    r32, st32, amb32 = _run(lib, monkeypatch, call, ["BOSS_SCREEN_NO_RESEED"])
    rrs, strs, ambrs = _run(lib, monkeypatch, call, [])
    for r in (r64, r32, rrs):
        assert key(r) == key(ref)
    assert st32 == st64, (st32, st64)
    if st32[0] == 1:   # the raw pool holds the pool plus the ambiguous candidates that the refinement dropped
        assert st32[2] <= amb32[1] <= st32[2] + amb32[0], (st32, amb32)
        assert strs[2] <= st32[2], (strs, st32)
        assert ambrs == amb32, (ambrs, amb32)
    return st32, amb32, strs


def _pair_key(r):
    return (_bits(r[0]), int(r[1]))


def _topk_key(r):
    tv, ti = r
    return ([_bits(v) for v in tv], [int(i) for i in ti])


@pytest.fixture(scope="module")
def bench_problem(lib):
    X, Y, ls, amp, ns = make_problem(2048, 8, seed=1002)
    gp = lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], lib.KERNEL_MATERN52)
    Xs = np.random.default_rng(7).random((8, M))
    yield gp, float(np.max(Y[0])), Xs
    gp.free()


def test_pool_bench_problem_all_input_forms(lib, monkeypatch, bench_problem):
    import torch
    gp, best, Xs = bench_problem
    st, amb, strs = _tiers(lib, monkeypatch,
                           lambda: lib.ei_score([gp], 1, 1, Xs, [1.0], best, None, want_acq=False)[1:], _pair_key)
    assert st[0] == 1 and strs[0] == 1
    print(f"pool {st[2]}, ambiguous {amb[0]}, after re-seed {strs[2]}")
    pinned = torch.empty((M, 8), dtype=torch.float64, pin_memory=True)
    pinned.copy_(torch.from_numpy(np.ascontiguousarray(Xs.T)))
    _tiers(lib, monkeypatch, lambda: lib.ei_score([gp], 1, 1, pinned.numpy().T, [1.0], best, None, want_acq=False)[1:],
           _pair_key)
    dev = pinned.cuda()
    torch.cuda.synchronize()
    _tiers(lib, monkeypatch, lambda: lib.ei_score_dev([gp], 1, 1, dev.data_ptr(), M, [1.0], best, None), _pair_key)


@pytest.mark.parametrize("k", [1, 7, 128])
def test_pool_topk(lib, monkeypatch, bench_problem, k):
    gp, best, Xs = bench_problem
    _tiers(lib, monkeypatch, lambda: lib.ei_score_topk([gp], 1, 1, Xs, [1.0], best, None, k), _topk_key)


def test_pool_bi_two_outputs_prior_mean(lib, monkeypatch):
    n, d = 2048, 8
    X, Y, ls, amp, ns = make_problem(n, d, seed=43, y_dim=2)
    gps = [lib.gp_fit(X, Y[i], ls[i], amp[i], ns[i], lib.KERNEL_MATERN52) for i in range(2)]
    rng = np.random.default_rng(44)
    Xs = rng.random((d, M)) * 1.2 - 0.1
    coefs = np.array([1.0, -0.5])
    best = float(np.max(coefs @ Y))
    cm = (rng.random(M) > 0.2).astype(np.uint8)
    pm = 0.05 * rng.standard_normal((2, M))
    lb, ub = np.zeros(d), np.ones(d)
    _tiers(lib, monkeypatch, lambda: lib.ei_score(gps, 2, 1, Xs, coefs, best, None, lb=lb, ub=ub, cons_mask=cm,
                                                  prior_mean_s=pm, want_acq=False)[1:], _pair_key)
    _tiers(lib, monkeypatch, lambda: lib.ei_score_topk(gps, 2, 1, Xs, coefs, best, None, 7, lb=lb, ub=ub,
                                                       cons_mask=cm, prior_mean_s=pm), _topk_key)
    for g in gps:
        g.free()
    X, Y, ls, amp, ns = make_problem(512, 5, seed=41)
    gps = [lib.gp_fit(X, Y[0], ls[0] * f, amp[0] * g, ns[0], lib.KERNEL_MATERN52)
           for f, g in ((1.0, 1.0), (0.8, 1.2), (1.3, 0.9))]
    Xs = np.random.default_rng(42).random((5, M))
    _tiers(lib, monkeypatch, lambda: lib.ei_score(gps, 1, 3, Xs, [1.0], float(np.max(Y[0])), None, want_acq=False)[1:],
           _pair_key)
    for g in gps:
        g.free()


def test_pool_generators_nan_and_fallback(lib, monkeypatch):
    n, d = 2048, 8
    X, Y, ls, amp, ns = make_problem(n, d, seed=47)
    gp = lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], lib.KERNEL_MATERN52)
    best = float(np.max(Y[0]))
    _tiers(lib, monkeypatch,
           lambda: lib.ei_score_uniform([gp], 1, 1, 99, M, np.zeros(d), np.ones(d), [1.0], best, None)[1:3], _pair_key)
    count = np.array([5, 5, 5, 5, 5, 5, 5, 4])
    _tiers(lib, monkeypatch,
           lambda: lib.ei_score_grid([gp], 1, 1, np.zeros(d), 1.0 / (count - 1), count, [1.0], best, None)[1:3],
           _pair_key)
    Xs = np.random.default_rng(48).random((d, M))
    Xs[1, [150_001, 90_000, 150_000]] = np.nan
    st, amb, _ = _tiers(lib, monkeypatch,
                        lambda: lib.ei_score([gp], 1, 1, Xs, [1.0], best, None, want_acq=False)[1:], _pair_key)
    assert st[0] == 1 and amb[0] >= 2, (st, amb)   # the NaN candidates after the first chunk are ambiguous
    gp.free()
    X, Y, ls, amp, ns = make_problem(256, 4, seed=46)
    gp = lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], lib.KERNEL_MATERN52)
    Xs = np.tile(np.full((4, 1), 0.37), (1, M))
    st, _, _ = _tiers(lib, monkeypatch,
                      lambda: lib.ei_score([gp], 1, 1, Xs, [1.0], float(np.max(Y[0])), None, want_acq=False)[1:],
                      _pair_key)
    assert st[0] == 2, st
    gp.free()
