"""The variance tier of argmax screening (DESIGN.md 2.9): before the re-seeded pool is scored exactly, each pool row is
bounded by EI at a^2 - S1, S1 the sum of squares of the first row block of V = W K* (the first 128 training points),
and only rows whose bound reaches the re-seeded threshold go on.

- The bench problem (2 Mi candidates resident, pinned and pageable; top-k with k in {1, 7, 128}) and a 2-output BI call
  with prior means and a constraint mask: pairs and lists bit-identical to the unscreened call, the screening counters
  unchanged (5 491 ambiguous, raw pool 20 751, re-seeded pool 2 083 on the bench problem), survivors <= pool.
- On 65 536 candidates of the bench problem, the tier's bound evaluated on the host from the first row block is at
  least every candidate's exact device score.
"""
import numpy as np
import pytest
from scipy.linalg import solve_triangular
from scipy.special import erfc

from oracle import boss_oracle as O
from tests.util_problems import make_problem

pytestmark = pytest.mark.gpu

M = 1 << 21


def _bits(v):
    return int(np.float64(v).view(np.int64))


@pytest.fixture(scope="module")
def bench(lib):
    import torch
    X, Y, ls, amp, ns = make_problem(2048, 8, seed=1002)
    gp = lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], lib.KERNEL_MATERN52)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(2002)
    dev = torch.rand((M, 8), dtype=torch.float64, device="cuda", generator=gen)   # bench.py's candidates
    torch.cuda.synchronize()
    yield gp, dev, float(np.max(Y[0])), (X, Y, ls, amp, ns)
    gp.free()


def _screened_vs_full(lib, monkeypatch, call):
    monkeypatch.delenv("BOSS_NO_SCREEN", raising=False)
    scr = call()
    counters = (lib.dbg_screen_stats(), lib.dbg_screen_ambiguous(), lib.dbg_screen_var())
    monkeypatch.setenv("BOSS_NO_SCREEN", "1")
    full = call()
    monkeypatch.delenv("BOSS_NO_SCREEN", raising=False)
    return scr, full, counters


def test_bench_problem_resident_pinned_pageable(lib, monkeypatch, bench):
    import torch
    gp, dev, best, _ = bench
    pinned = torch.empty((M, 8), dtype=torch.float64, pin_memory=True)
    pinned.copy_(dev.cpu())
    pageable = pinned.numpy().copy()
    calls = {
        "resident": lambda: lib.ei_score_dev([gp], 1, 1, dev.data_ptr(), M, [1.0], best, None),
        "pinned": lambda: lib.ei_score([gp], 1, 1, pinned.numpy().T, [1.0], best, None, want_acq=False)[1:],
        "pageable": lambda: lib.ei_score([gp], 1, 1, pageable.T, [1.0], best, None, want_acq=False)[1:],
    }
    for name, call in calls.items():
        scr, full, (st, amb, var) = _screened_vs_full(lib, monkeypatch, call)
        print(name, st, amb, var)
        assert (_bits(scr[0]), int(scr[1])) == (_bits(full[0]), int(full[1])), name
        assert st == (1, M, 2083) and amb == (5491, 20751), (name, st, amb)
        assert var[0] == 2083 and 1 <= var[1] <= var[0], (name, var)


# k = 128: the 128th best seed score lets 20 827 of the first chunk's 75 776 candidates through, more than a quarter,
# so the call falls back to the full path and the tier does not run
@pytest.mark.parametrize("k,state", [(1, 1), (7, 1), (128, 2)])
def test_bench_problem_topk(lib, monkeypatch, bench, k, state):
    gp, dev, best, _ = bench
    scr, full, (st, _, var) = _screened_vs_full(
        lib, monkeypatch, lambda: lib.ei_score_topk_dev([gp], 1, 1, dev.data_ptr(), M, [1.0], best, None, k))
    assert st[0] == state, st
    assert np.array_equal(scr[0].view(np.int64), full[0].view(np.int64))
    assert np.array_equal(scr[1], full[1])
    if state == 1:
        assert k <= var[1] <= var[0] == st[2], (var, st)
    else:
        assert var == (0, 0), var


def test_bi_two_outputs_prior_mean_mask(lib, monkeypatch):
    monkeypatch.setenv("BOSS_SCREEN_MIN_M", "4096")
    n, d, m = 512, 5, 300_000
    X, Y, ls, amp, ns = make_problem(n, d, seed=83, y_dim=2)
    gps = [lib.gp_fit(X, Y[i], ls[i] * f, amp[i], ns[i], lib.KERNEL_MATERN52) for f in (1.0, 0.8) for i in range(2)]
    rng = np.random.default_rng(84)
    Xs = rng.random((d, m))
    pm = 0.05 * rng.standard_normal((2, m))
    cm = (rng.random(m) > 0.1).astype(np.uint8)
    best = float(np.max(Y[0] - 0.5 * Y[1]))
    scr, full, (st, _, var) = _screened_vs_full(lib, monkeypatch, lambda: lib.ei_score(
        gps, 2, 2, Xs, [1.0, -0.5], best, None, cons_mask=cm, prior_mean_s=pm, want_acq=False)[1:])
    assert st[0] == 1, st
    assert (_bits(scr[0]), int(scr[1])) == (_bits(full[0]), int(full[1]))
    assert var[0] == st[2] and 1 <= var[1] <= var[0], (var, st)
    for g in gps:
        g.free()


def test_tier_bound_holds(lib, monkeypatch, bench):
    """EI at a^2 - S1 (first 128 training points, host FP64) with the host mean bounds every exact device score."""
    gp, dev, best, (X, Y, ls, amp, ns) = bench
    m = 65536
    Xs = dev[:m].cpu().numpy().T.copy()
    monkeypatch.setenv("BOSS_NO_SCREEN", "1")
    acq = lib.ei_score([gp], 1, 1, Xs, [1.0], best, None)[0]
    post = O.posterior_fit(X, Y[0], ls[0], amp[0], ns[0], O.KERNEL_MATERN52)
    mu = np.empty(m)
    for i in range(0, m, 8192):
        mu[i:i + 8192] = O.kernel_matrix(X, Xs[:, i:i + 8192], post.ls, post.amp, O.KERNEL_MATERN52).T @ post.alpha_w
    K1 = O.kernel_matrix(X[:, :128], Xs, post.ls, post.amp, O.KERNEL_MATERN52)
    V1 = solve_triangular(post.U[:128, :128].T, K1, lower=True)   # the first row block of W K* = L11^-1 K*_1
    var = np.maximum(post.amp ** 2 - (V1 * V1).sum(0) + 1e-18, 0.0)
    sd = np.sqrt(var)
    z = (mu - best) / sd
    bound = (mu - best) * 0.5 * erfc(-z / np.sqrt(2.0)) + sd * np.exp(-0.5 * z * z) / np.sqrt(2.0 * np.pi)
    ok = bound >= acq * (1.0 - 1e-9) - 1e-300
    assert ok.all(), (np.count_nonzero(~ok), float(np.max((acq - bound)[~ok])))
    assert np.count_nonzero(bound < 0.5 * bound.max()) > 0   # the bound is not the prior-variance one everywhere
