"""Device-resident screened calls run the FP32 mean tier's pass over every candidate after the first chunk on a side
stream, beside the first chunk's FP64 means, seed batch and threshold (DESIGN.md 2.9).  The pass writes bounds only;
the counts come after the join.  Results, pools and verdicts must be those of the single-stream order:

- the bench problem's pair (with the pool counts of the host-staged path), top-k lists for k in {1, 7, 128} and a
  2-output BI call with prior means and a constraint mask equal the unscreened call bit for bit;
- identical candidates fall back to the full path behind the side pass and return its pair;
- 20 repeated resident calls, with timing mode on and off, return the same bits and pool counts.
"""
import numpy as np
import pytest

from tests.util_problems import make_problem

pytestmark = pytest.mark.gpu

M = 300_000   # the first chunk (75 776) and one side-stream piece of 224 224 candidates


def _bits(v):
    return int(np.float64(v).view(np.int64))


def _dev(a):
    import torch
    t = torch.from_numpy(np.ascontiguousarray(a)).cuda()
    torch.cuda.synchronize()
    return t


def _both(lib, monkeypatch, call):
    monkeypatch.setenv("BOSS_SCREEN_MIN_M", "4096")
    monkeypatch.delenv("BOSS_NO_SCREEN", raising=False)
    scr = call()
    st = lib.dbg_screen_stats()
    amb = lib.dbg_screen_ambiguous()
    monkeypatch.setenv("BOSS_NO_SCREEN", "1")
    full = call()
    monkeypatch.delenv("BOSS_NO_SCREEN", raising=False)
    return scr, full, st, amb


@pytest.fixture(scope="module")
def bench_gp(lib):
    X, Y, ls, amp, ns = make_problem(2048, 8, seed=1002)
    gp = lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], lib.KERNEL_MATERN52)
    Xs = np.random.default_rng(81).random((8, M))
    yield gp, Xs, float(np.max(Y[0]))
    gp.free()


def test_argmax_matches_host_paths_and_full(lib, monkeypatch, bench_gp):
    gp, Xs, best = bench_gp
    dev = _dev(Xs.T)
    scr, full, st, amb = _both(lib, monkeypatch,
                               lambda: lib.ei_score_dev([gp], 1, 1, dev.data_ptr(), M, [1.0], best, None))
    assert st[0] == 1, st
    assert (_bits(scr[0]), scr[1]) == (_bits(full[0]), full[1])
    hscr, _, hst, hamb = _both(lib, monkeypatch,
                               lambda: lib.ei_score([gp], 1, 1, Xs, [1.0], best, None, want_acq=False)[1:])
    assert (_bits(hscr[0]), hscr[1]) == (_bits(scr[0]), scr[1])
    assert hst == st and hamb == amb, (hst, st, hamb, amb)


# k = 128: the 128th best seed score lets 22 752 of the first chunk's 75 776 candidates through, more than a quarter,
# so the call falls back to the full path behind the side stream's pass
@pytest.mark.parametrize("k,state", [(1, 1), (7, 1), (128, 2)])
def test_topk_matches_full(lib, monkeypatch, bench_gp, k, state):
    gp, Xs, best = bench_gp
    dev = _dev(Xs.T)
    scr, full, st, _ = _both(lib, monkeypatch,
                             lambda: lib.ei_score_topk_dev([gp], 1, 1, dev.data_ptr(), M, [1.0], best, None, k))
    assert st[0] == state, st
    assert np.array_equal(scr[0].view(np.int64), full[0].view(np.int64))
    assert np.array_equal(scr[1], full[1])


def test_bi_two_outputs_prior_mean_mask(lib, monkeypatch):
    n, d = 512, 5
    X, Y, ls, amp, ns = make_problem(n, d, seed=83, y_dim=2)
    gps = [lib.gp_fit(X, Y[i], ls[i] * f, amp[i], ns[i], lib.KERNEL_MATERN52) for f in (1.0, 0.8) for i in range(2)]
    rng = np.random.default_rng(84)
    Xs = rng.random((d, M))
    pm = 0.05 * rng.standard_normal((M, 2))
    cm = (rng.random(M) > 0.1).astype(np.uint8)
    dx, dpm, dcm = _dev(Xs.T), _dev(pm), _dev(cm)
    coefs = [1.0, -0.5]
    best = float(np.max(Y[0] - 0.5 * Y[1]))
    scr, full, st, _ = _both(lib, monkeypatch, lambda: lib.ei_score_dev(
        gps, 2, 2, dx.data_ptr(), M, coefs, best, None, prior_mean_ptr=dpm.data_ptr(), cons_mask_ptr=dcm.data_ptr()))
    assert st[0] == 1, st
    assert (_bits(scr[0]), scr[1]) == (_bits(full[0]), full[1])
    for g in gps:
        g.free()


def test_identical_candidates_fall_back(lib, monkeypatch):
    n, d = 256, 4
    X, Y, ls, amp, ns = make_problem(n, d, seed=46)
    gp = lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], lib.KERNEL_MATERN52)
    dev = _dev(np.full((M, d), 0.37))
    best = float(np.max(Y[0]))
    scr, full, st, _ = _both(lib, monkeypatch, lambda: lib.ei_score_dev([gp], 1, 1, dev.data_ptr(), M, [1.0], best, None))
    assert st[0] == 2 and st[1] == 75_776 and st[2] == 75_776, st
    assert (_bits(scr[0]), scr[1]) == (_bits(full[0]), full[1])
    gp.free()


@pytest.mark.parametrize("timing", [False, True])
def test_repeated_calls_identical(lib, monkeypatch, bench_gp, timing):
    gp, Xs, best = bench_gp
    dev = _dev(Xs.T)
    monkeypatch.setenv("BOSS_SCREEN_MIN_M", "4096")
    monkeypatch.delenv("BOSS_NO_SCREEN", raising=False)
    lib.set_timing(timing)
    try:
        seen = set()
        for _ in range(20):
            r = lib.ei_score_dev([gp], 1, 1, dev.data_ptr(), M, [1.0], best, None)
            seen.add((_bits(r[0]), int(r[1]), tuple(lib.dbg_screen_stats()), tuple(lib.dbg_screen_ambiguous())))
    finally:
        lib.set_timing(False)
    assert len(seen) == 1, seen
    assert next(iter(seen))[2][0] == 1
