"""The FP32 mean tier's fused kernel (screen_mean_bound_kernel, DESIGN.md 2.9) on device-resident candidates, where one
launch covers every candidate after the first chunk.

- On the bench problem without re-seed: the ambiguous count and the raw pool (keeps plus ambiguous, before the FP64
  refinement) that the per-chunk kernels gave (5 491 and 20 751), the refined pool equal to the FP64 tier's (17 832), and
  the unscreened pair.
- A 2-slice BI call, a call with NaN and far-outside-the-box candidates, and a call with more slices than one launch
  takes (screened with FP64 means): results equal the unscreened call bit for bit, pools those of the FP64 tier.
"""
import numpy as np
import pytest

from tests.util_problems import make_problem

pytestmark = pytest.mark.gpu

ENV = ("BOSS_NO_SCREEN", "BOSS_SCREEN_F64", "BOSS_SCREEN_NO_RESEED")


def _bits(v):
    return int(np.float64(v).view(np.int64))


def _run(lib, monkeypatch, call, env):
    for k in ENV:
        monkeypatch.delenv(k, raising=False)
    for k in env:
        monkeypatch.setenv(k, "1")
    r = call()
    return (_bits(r[0]), int(r[1])), lib.dbg_screen_stats(), lib.dbg_screen_ambiguous()


def _tiers(lib, monkeypatch, call):
    ref, st0, _ = _run(lib, monkeypatch, call, ["BOSS_NO_SCREEN"])
    r64, st64, amb64 = _run(lib, monkeypatch, call, ["BOSS_SCREEN_F64", "BOSS_SCREEN_NO_RESEED"])
    r32, st32, amb32 = _run(lib, monkeypatch, call, ["BOSS_SCREEN_NO_RESEED"])
    rrs, strs, _ = _run(lib, monkeypatch, call, [])
    assert st0[0] == 0
    assert r64 == ref and r32 == ref and rrs == ref, (ref, r64, r32, rrs)
    assert st32 == st64, (st32, st64)
    assert strs[2] <= st32[2]
    return st32, amb32, amb64


def _dev(Xs):
    import torch
    t = torch.from_numpy(np.ascontiguousarray(Xs.T)).cuda()
    torch.cuda.synchronize()
    return t


def test_bench_problem_counts(lib, monkeypatch):
    import torch
    X, Y, ls, amp, ns = make_problem(2048, 8, seed=1002)
    gp = lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], lib.KERNEL_MATERN52)
    M = 1 << 21
    gen = torch.Generator(device="cuda")
    gen.manual_seed(2002)
    Xs = torch.rand((M, 8), dtype=torch.float64, device="cuda", generator=gen)   # bench.py's candidates
    torch.cuda.synchronize()
    best = float(np.max(Y[0]))
    st, amb, amb64 = _tiers(lib, monkeypatch, lambda: lib.ei_score_dev([gp], 1, 1, Xs.data_ptr(), M, [1.0], best, None))
    print(f"bench call: stats {st}, ambiguous {amb[0]}, raw pool {amb[1]}")
    assert st[0] == 1
    assert amb64[0] == 0
    assert (amb[0], amb[1], st[2]) == (5491, 20751, 17832), (amb, st)
    gp.free()


def test_bi_two_slices_dev(lib, monkeypatch):
    monkeypatch.setenv("BOSS_SCREEN_MIN_M", "4096")
    n, d, M = 1024, 6, 300_000
    X, Y, ls, amp, ns = make_problem(n, d, seed=51)
    gps = [lib.gp_fit(X, Y[0], ls[0] * f, amp[0] * g, ns[0], lib.KERNEL_MATERN32) for f, g in ((1.0, 1.0), (0.7, 1.3))]
    Xs = _dev(np.random.default_rng(52).random((d, M)))
    st, amb, _ = _tiers(lib, monkeypatch,
                        lambda: lib.ei_score_dev(gps, 1, 2, Xs.data_ptr(), M, [1.0], float(np.max(Y[0])), None))
    assert st[0] == 1, st
    for g in gps:
        g.free()


def test_nan_and_far_outside_dev(lib, monkeypatch):
    monkeypatch.setenv("BOSS_SCREEN_MIN_M", "4096")
    n, d, M = 2048, 8, 400_000
    X, Y, ls, amp, ns = make_problem(n, d, seed=47)
    gp = lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], lib.KERNEL_MATERN52)
    Xs = np.random.default_rng(48).random((d, M))
    Xs[1, [150_001, 90_000, 399_999]] = np.nan
    Xs[:, 200_000:200_300] = 1e6   # far outside the box: mean ~ 0, E tiny
    Xs[3, 250_000] = -1e30
    dev = _dev(Xs)
    st, amb, _ = _tiers(lib, monkeypatch,
                        lambda: lib.ei_score_dev([gp], 1, 1, dev.data_ptr(), M, [1.0], float(np.max(Y[0])), None))
    assert st[0] == 1 and amb[0] >= 3, (st, amb)   # the NaN candidates after the first chunk are ambiguous
    gp.free()


def test_more_slices_than_one_launch_dev(lib, monkeypatch):
    """17 BI samples: more than the fused kernel takes, so the call screens with FP64 means (no ambiguous band)."""
    monkeypatch.setenv("BOSS_SCREEN_MIN_M", "4096")
    n, d, M = 256, 4, 200_000
    X, Y, ls, amp, ns = make_problem(n, d, seed=53)
    gps = [lib.gp_fit(X, Y[0], ls[0] * (0.8 + 0.025 * k), amp[0], ns[0], lib.KERNEL_SE) for k in range(17)]
    Xs = _dev(np.random.default_rng(54).random((d, M)))
    st, amb, _ = _tiers(lib, monkeypatch,
                        lambda: lib.ei_score_dev(gps, 1, 17, Xs.data_ptr(), M, [1.0], float(np.max(Y[0])), None))
    if st[0] == 1:
        assert amb[0] == 0, amb
    for g in gps:
        g.free()
