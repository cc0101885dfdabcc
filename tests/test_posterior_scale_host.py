"""CPU checks of tests/posterior_scale_oracle.py: the long-double posterior and x-gradients against 40-digit mpmath, the
FP64 reference against the long-double values at eight blocks, the sensitivity of the device comparisons to one
wrong tile, block or lengthscale, and the mirror of the scoring call's chunk and path choice."""
import numpy as np
import pytest

from oracle import boss_oracle as OB
from tests import posterior_scale_oracle as PS
from tests.kernels_more_oracle import KERNEL_MATERN12, RQ
from tests.util_problems import make_problem

ALL_KERNELS = [OB.KERNEL_SE, OB.KERNEL_MATERN32, OB.KERNEL_MATERN52, KERNEL_MATERN12, RQ(0.5), RQ(3.0)]
IDS = ["se", "matern32", "matern52", "matern12", "rq0.5", "rq3"]


def _candidates(X, M, seed):
    """M random candidates in the unit box, the first two on training points."""
    Xs = np.random.default_rng(seed).random((X.shape[0], M))
    Xs[:, 0] = X[:, 3]
    Xs[:, 1] = X[:, -1]
    return Xs


@pytest.mark.parametrize("kernel", ALL_KERNELS, ids=IDS)
def test_longdouble_posterior_gradient_matches_mpmath(kernel):
    pytest.importorskip("mpmath")
    n, d = 10, 3
    X, Y, ls, amp, ns = make_problem(n, d, seed=60)
    X[1] = np.round(X[1] * 3) + 0.1 * X[1]               # a discrete dimension: rounded to 0..3
    mask = np.array([False, True, False])
    Xs = _candidates(X, 4, seed=61)
    Xs[1, 2:] = [0.8, 2.3]
    for m in (None, mask):
        got = PS.adjudicator_post_grad_longdouble(X, Y[0], ls[0], amp[0], ns[0], kernel, Xs, m)
        ref = PS.mp_post_grad(X, Y[0], ls[0], amp[0], ns[0], kernel, Xs, m)
        for name, g, r in zip(("mu", "var", "dmu", "dvar"), got, ref):
            scale = np.max(np.abs(r), axis=-1, keepdims=True)
            assert np.all(np.abs(g - r) <= 1e-15 * scale), (name, g, r)
        if m is not None:
            assert np.all(got[2][1] == 0.0) and np.all(got[3][1] == 0.0)
            assert np.any(got[2][0] != 0.0)


# n = 1024, d = 8 (DP 8, eight full blocks) and n = 769, d = 32 (DP 32, one live row in the last block)
SHAPES = [(1024, 8, 1024), (769, 32, 769)]


@pytest.mark.parametrize("n,d,seed", SHAPES, ids=["n1024_d8", "n769_d32"])
@pytest.mark.parametrize("kernel", ALL_KERNELS, ids=IDS)
def test_fp64_reference_is_far_inside_every_ratio(kernel, n, d, seed):
    """Justifies the FP64 oracle as the reference for device results: against the long-double values it uses at most a tenth of
    each comparison's tolerance."""
    X, Y, ls, amp, ns = make_problem(n, d, seed=seed)
    Xs = _candidates(X, 48, seed=seed + 1)
    Om = PS.reference(kernel)
    post = Om.posterior_fit(X, Y[0], ls[0], amp[0], ns[0], kernel)
    mu, var, dmu, dvar, st = Om.mean_var_grad(post, Xs)
    assert np.all(st == 0)
    truth = PS.adjudicator_post_grad_longdouble(X, Y[0], ls[0], amp[0], ns[0], kernel, Xs)
    r = PS.post_grad_ratios((mu, var, dmu, dvar), truth, PS.post_bounds(X, Y[0], ls[0], amp[0], ns[0], kernel, Xs))
    print(f"n={n} d={d} {kernel}: FP64 reference vs long double, ratio to tolerance: "
          + ", ".join(f"{k} {v:.2e}" for k, v in r.items()))
    assert max(r.values()) <= 0.1, r


@pytest.mark.parametrize("kernel", [OB.KERNEL_MATERN52, KERNEL_MATERN12, RQ(0.5)], ids=["matern52", "matern12", "rq0.5"])
def test_comparisons_see_every_tile(kernel):
    """n = 1000: 8 blocks, the last ragged with 104 live rows.  A missing tile or block is rejected by >= 1e6x, a 1e-6
    error in one 1/l by >= 10x."""
    n, d = 1000, 4
    X, Y, ls, amp, ns = make_problem(n, d, seed=1000)
    Xs = _candidates(X, 40, seed=1001)
    args = (X, Y[0], ls[0], amp[0], ns[0], kernel, Xs)
    Om = PS.reference(kernel)
    post = Om.posterior_fit(*args[:6])
    mu, var, dmu, dvar, _ = Om.mean_var_grad(post, Xs)
    true = (mu, var, dmu, dvar)
    bounds = PS.post_bounds(*args)
    assert max(PS.post_grad_ratios(PS.perturbed_post_grad(*args), true, bounds).values()) <= 0.1   # unperturbed

    def worst(**kw):
        return max(PS.post_grad_ratios(PS.perturbed_post_grad(*args, **kw), true, bounds).values())

    nblk = (n + 127) // 128
    tiles = [worst(zero_w_tile=(bi, bj)) for bi in range(nblk) for bj in range(bi)]
    assert len(tiles) == 28
    others = dict(ks_tail=worst(zero_ks_tail=17), wt_last_rows=worst(drop_wt_last_rows=True),
                  invl=min(worst(dinvl=(j, 1e-6)) for j in range(d)))
    print(f"{kernel}: smallest rejection over 28 zeroed W tiles {min(tiles):.3g}; "
          + ", ".join(f"{k} {v:.3g}" for k, v in others.items()))
    assert min(tiles) >= 1e6 and others["ks_tail"] >= 1e6 and others["wt_last_rows"] >= 1e6   # structural: far outside
    assert others["invl"] >= 10                                   # 1e-6 relative in one dimension against 1e-8


def _paths(plan):
    return [(p["chunk"], p["slice"], p["path"], p["nsp32"] if p["path"] == "narrow" else p["nsp"]) for p in plan["passes"]]


def test_score_plan_chunks():
    assert PS.chunk_capacity([2048], 10 ** 6, 8, False) == (75776, False)    # 592 candidate blocks
    assert PS.chunk_capacity([2048], 10 ** 6, 8, True) == (37888, True)      # 296 with gradients
    assert PS.chunk_capacity([4096], 10 ** 6, 4, False) == (75776, False)
    assert PS.chunk_capacity([8192], 10 ** 6, 4, False) == (512 // 148 * 148 * 128, False)   # the 4 GiB K*^T budget
    assert PS.chunk_capacity([2048], 8192, 8, False) == (8192, True)         # V^T kept up to 8192 candidates
    assert PS.chunk_capacity([2048], 8193, 8, False) == (8320, False)
    assert PS.chunk_capacity([2048] * 16, 10 ** 6, 32, False, pgrad=True)[0] == 246 * 128   # the PGRAD slot
    assert PS.chunk_capacity([2048] * 16, 10 ** 6, 8, False, pgrad=True)[0] == 37888
    assert PS.chunk_capacity([128, 2049], 100, 3, False) == (128, True)      # sized by the largest slice


def test_score_plan_paths():
    # value-only calls at n = 2048: quarter, wide with splits, wide fused, and the narrow tail of a two-chunk call
    assert _paths(PS.score_plan(2048, 1, 8, False)) == [(0, 0, "quarter", 16)]
    assert _paths(PS.score_plan(2048, 8192, 8, False)) == [(0, 0, "quarter", 2)]
    assert _paths(PS.score_plan(2048, 8193, 8, False)) == [(0, 0, "wide_split", 2)]
    assert _paths(PS.score_plan(2048, 37888, 8, False)) == [(0, 0, "wide_fused", 1)]
    assert _paths(PS.score_plan(2048, 37889, 8, False)) == [(0, 0, "wide_split", 8)]
    assert _paths(PS.score_plan(2048, 75776 + 300, 8, False)) == [(0, 0, "wide_fused", 1), (1, 0, "narrow", 8)]
    assert _paths(PS.score_plan(2048, 75776 + 5000, 8, False)) == [(0, 0, "wide_fused", 1), (1, 0, "narrow", 8)]
    assert _paths(PS.score_plan(4096, 75777, 4, False)) == [(0, 0, "wide_fused", 1), (1, 0, "narrow", 32)]
    # with gradients: the chunk is 296 blocks, V^T always exists and the tail goes through quarter
    assert _paths(PS.score_plan(2048, 37889, 8, True)) == [(0, 0, "wide_fused", 1), (1, 0, "quarter", 16)]
    assert _paths(PS.score_plan(2048, 8193, 8, True)) == [(0, 0, "quarter", 2)]
    assert _paths(PS.score_plan(2048, 8513, 8, True)) == [(0, 0, "wide_split", 2)]
    # one block: never quarter; a one-candidate tail still goes through narrow
    assert _paths(PS.score_plan(64, 75777, 3, False)) == [(0, 0, "wide_fused", 1), (1, 0, "narrow", 1)]
    assert _paths(PS.score_plan(2048, 75776 + 5000, 8, True)) == [(0, 0, "wide_fused", 1), (1, 0, "wide_fused", 1),
                                                                   (2, 0, "quarter", 8)]
    # several slices: only the last fuses; mixed block counts pick per slice
    assert [p["path"] for p in PS.score_plan(2048, 37888, 8, False, nsl=3)["passes"]] == ["wide_split"] * 2 + ["wide_fused"]
    assert _paths(PS.score_plan([128, 129], 8, 3, False)) == [(0, 0, "narrow", 1), (0, 1, "quarter", 2)]
    # forced paths: quarter needs V^T; BOSS_UNFUSED_SCORE leaves every pass unfused
    assert _paths(PS.score_plan(2048, 37888, 8, False, path="quarter")) == [(0, 0, "wide_fused", 1)]
    assert _paths(PS.score_plan(2048, 8192, 8, False, path="wide")) == [(0, 0, "wide_split", 2)]
    assert _paths(PS.score_plan(2048, 37888, 8, True, path="narrow")) == [(0, 0, "narrow", 1)]
    assert _paths(PS.score_plan(2048, 37888, 8, False, unfused=True)) == [(0, 0, "wide_split", 1)]


def test_score_plan_counts_and_edges():
    p = PS.score_plan(2048, 75776 + 300, 8, False, nsl=2)     # two chunks x two slices; only slice 1 may fuse
    assert PS.plan_counts(p) == dict(wide_fused=1, wide_split=1, narrow=2, quarter=0, xgrad=0)
    assert PS.chunk_edges(p, 75776 + 300) == [0, 75775, 75776, 76075]
    p = PS.score_plan(2048, 75776 + 300, 8, True, nsl=2)      # three chunks of at most 296 blocks
    assert PS.plan_counts(p) == dict(wide_fused=2, wide_split=2, narrow=0, quarter=2, xgrad=6)
    assert PS.chunk_edges(p, 75776 + 300) == [0, 37887, 37888, 75775, 75776, 76075]
