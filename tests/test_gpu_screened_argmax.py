"""Argmax screening (DESIGN.md 2.9): a call that wants only the (best value, index) pair of the closed-form EI bounds
every candidate by its EI at the prior standard deviation and scores exactly only the candidates whose bound can still
beat the best of a seed batch.  The pair must be bit-identical to the unscreened call (BOSS_NO_SCREEN=1) for every
input form, and the debug counters show whether screening ran or fell back."""
import numpy as np
import pytest

from tests.util_problems import make_problem

pytestmark = pytest.mark.gpu

M = 200_000   # several 75 776-candidate chunks at n <= 4096: the pool collects survivors of more than one chunk
# The bound is the EI at the prior variance, so it separates where the posterior is much tighter than the prior: the
# screened tests use bench.py's shape (n = 2048, d = 8); small, low-dimensional problems may fall back.


def _bits(v):
    return int(np.array(v, dtype=np.float64).view(np.int64))


def _screened_vs_full(lib, monkeypatch, call):
    """Runs call() screened and with BOSS_NO_SCREEN=1; asserts equal pairs; returns the screened call's counters."""
    monkeypatch.setenv("BOSS_SCREEN_MIN_M", "4096")
    monkeypatch.delenv("BOSS_NO_SCREEN", raising=False)
    bv1, bi1 = call()
    st = lib.dbg_screen_stats()
    monkeypatch.setenv("BOSS_NO_SCREEN", "1")
    bv0, bi0 = call()
    assert lib.dbg_screen_stats()[0] == 0
    assert (_bits(bv1), bi1) == (_bits(bv0), bi0), (bv1, bi1, bv0, bi0)
    return st


def _assert_screened(st, m=M):
    state, bounded, surv = st
    assert state == 1 and bounded == m, st
    assert 1 <= surv < m // 10, st


def _fit(lib, n, d, seed, y_dim=1):
    X, Y, ls, amp, ns = make_problem(n, d, seed=seed, y_dim=y_dim)
    gps = [lib.gp_fit(X, Y[i], ls[i], amp[i], ns[i], lib.KERNEL_MATERN52) for i in range(y_dim)]
    return X, Y, ls, amp, ns, gps


@pytest.fixture(scope="module")
def bench_problem(lib):
    X, Y, ls, amp, ns, gps = _fit(lib, 2048, 8, 1002)
    Xs = np.random.default_rng(7).random((8, M))
    yield gps[0], float(np.max(Y[0])), Xs
    gps[0].free()


def test_bench_problem_host_pageable(lib, monkeypatch, bench_problem):
    gp, best, Xs = bench_problem
    st = _screened_vs_full(lib, monkeypatch, lambda: lib.ei_score([gp], 1, 1, Xs, [1.0], best, None, want_acq=False)[1:])
    _assert_screened(st)


def test_bench_problem_host_pinned_and_device(lib, monkeypatch, bench_problem):
    import torch
    gp, best, Xs = bench_problem
    pinned = torch.empty((M, 8), dtype=torch.float64, pin_memory=True)
    pinned.copy_(torch.from_numpy(np.ascontiguousarray(Xs.T)))
    st = _screened_vs_full(lib, monkeypatch,
                           lambda: lib.ei_score([gp], 1, 1, pinned.numpy().T, [1.0], best, None, want_acq=False)[1:])
    _assert_screened(st)
    dev = pinned.cuda()
    torch.cuda.synchronize()
    st = _screened_vs_full(lib, monkeypatch, lambda: lib.ei_score_dev([gp], 1, 1, dev.data_ptr(), M, [1.0], best, None))
    _assert_screened(st)
    # the host and device forms agree with each other too
    monkeypatch.delenv("BOSS_NO_SCREEN", raising=False)
    assert lib.ei_score_dev([gp], 1, 1, dev.data_ptr(), M, [1.0], best, None)[1] == \
        lib.ei_score([gp], 1, 1, Xs, [1.0], best, None, want_acq=False)[2]


def test_bi_samples(lib, monkeypatch):
    n, d = 512, 5
    X, Y, ls, amp, ns = make_problem(n, d, seed=41)
    gps = [lib.gp_fit(X, Y[0], ls[0] * f, amp[0] * g, ns[0], lib.KERNEL_MATERN52)
           for f, g in ((1.0, 1.0), (0.8, 1.2), (1.3, 0.9))]
    Xs = np.random.default_rng(42).random((d, M))
    best = float(np.max(Y[0]))
    st = _screened_vs_full(lib, monkeypatch, lambda: lib.ei_score(gps, 1, 3, Xs, [1.0], best, None, want_acq=False)[1:])
    _assert_screened(st)


def test_two_outputs_coefs_ymax_bounds_mask_prior_mean(lib, monkeypatch):
    n, d = 2048, 8
    X, Y, ls, amp, ns, gps = _fit(lib, n, d, 43, y_dim=2)
    rng = np.random.default_rng(44)
    Xs = rng.random((d, M)) * 1.2 - 0.1            # some candidates outside [0, 1]^d
    coefs = np.array([1.0, -0.5])
    y_max = np.array([np.inf, float(np.quantile(Y[1], 0.8))])
    best = float(np.max(coefs @ Y))
    cm = (rng.random(M) > 0.2).astype(np.uint8)
    pm = 0.05 * rng.standard_normal((2, M))
    lb, ub = np.zeros(d), np.ones(d)
    # the bound leaves PoF out: with a tight y_max the exact scores sit far below it and the call may fall back
    st = _screened_vs_full(lib, monkeypatch, lambda: lib.ei_score(gps, 2, 1, Xs, coefs, best, y_max, want_acq=False)[1:])
    assert st[0] in (1, 2), st
    st = _screened_vs_full(lib, monkeypatch, lambda: lib.ei_score(gps, 2, 1, Xs, coefs, best, y_max, lb=lb, ub=ub,
                                                                  cons_mask=cm, prior_mean_s=pm, want_acq=False)[1:])
    assert st[0] in (1, 2), st
    st = _screened_vs_full(lib, monkeypatch, lambda: lib.ei_score(gps, 2, 1, Xs, coefs, best, None, lb=lb, ub=ub,
                                                                  cons_mask=cm, want_acq=False)[1:])
    _assert_screened(st)
    st = _screened_vs_full(lib, monkeypatch, lambda: lib.ei_score(gps, 2, 1, Xs, coefs, best, None, lb=lb, ub=ub,
                                                                  cons_mask=cm, prior_mean_s=pm, want_acq=False)[1:])
    _assert_screened(st)


def test_generators(lib, monkeypatch):
    n, d = 2048, 8
    X, Y, ls, amp, ns, gps = _fit(lib, n, d, 45)
    best = float(np.max(Y[0]))
    count = np.array([5, 5, 5, 5, 5, 5, 5, 4])
    lo, step = np.zeros(d), 1.0 / (count - 1)
    st = _screened_vs_full(lib, monkeypatch,
                           lambda: lib.ei_score_grid(gps, 1, 1, lo, step, count, [1.0], best, None)[1:3])
    assert st[0] in (1, 2), st   # the first chunk of a grid is one corner of the box: the seed may not separate there
    st = _screened_vs_full(lib, monkeypatch,
                           lambda: lib.ei_score_uniform(gps, 1, 1, 99, M, np.zeros(d), np.ones(d), [1.0], best, None)[1:3])
    _assert_screened(st)


def test_identical_candidates_fall_back(lib, monkeypatch):
    """Every bound ties, so every candidate survives the first chunk: the call falls back to the full path."""
    n, d = 256, 4
    X, Y, ls, amp, ns, gps = _fit(lib, n, d, 46)
    Xs = np.tile(np.full((d, 1), 0.37), (1, M))
    best = float(np.max(Y[0]))
    st = _screened_vs_full(lib, monkeypatch, lambda: lib.ei_score(gps, 1, 1, Xs, [1.0], best, None, want_acq=False)[1:])
    assert st[0] == 2 and st[1] == 75_776 and st[2] == 75_776, st


def test_nan_candidates(lib, monkeypatch):
    """NaN bounds are kept and sort last among the seeds; the pair still matches the full path."""
    n, d = 2048, 8
    X, Y, ls, amp, ns, gps = _fit(lib, n, d, 47)
    Xs = np.random.default_rng(48).random((d, M))
    Xs[1, [150_001, 90_000, 150_000]] = np.nan
    best = float(np.max(Y[0]))
    st = _screened_vs_full(lib, monkeypatch, lambda: lib.ei_score(gps, 1, 1, Xs, [1.0], best, None, want_acq=False)[1:])
    _assert_screened(st)


def test_not_screened_below_threshold_or_with_outputs(lib, monkeypatch, bench_problem):
    gp, best, Xs = bench_problem
    monkeypatch.delenv("BOSS_NO_SCREEN", raising=False)
    monkeypatch.delenv("BOSS_SCREEN_MIN_M", raising=False)
    lib.ei_score([gp], 1, 1, Xs[:, :1], [1.0], best, None, want_acq=False)      # single point
    assert lib.dbg_screen_stats() == (0, 0, 0)
    lib.ei_score([gp], 1, 1, Xs[:, :60_000], [1.0], best, None, want_acq=False)  # below the default minimum
    assert lib.dbg_screen_stats() == (0, 0, 0)
    lib.ei_score([gp], 1, 1, Xs, [1.0], best, None, want_acq=True)              # per-candidate values requested
    assert lib.dbg_screen_stats() == (0, 0, 0)
    lib.ei_score([gp], 1, 1, Xs, [1.0], best, None, want_acq=False)
    assert lib.dbg_screen_stats()[0] == 1
