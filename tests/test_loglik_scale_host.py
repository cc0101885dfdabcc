"""CPU checks of tests/loglik_scale_oracle.py: the long-double gradient against 40-digit mpmath, the FP64 reference
against the long-double truth at n = 1024, the sensitivity of the GPU tests' gradient comparison, and the window /
stream-group mirror of loglik_core."""
import numpy as np
import pytest

from oracle import boss_oracle as OB
from tests import loglik_scale_oracle as LS
from tests.kernels_more_oracle import KERNEL_MATERN12, RQ
from tests.util_problems import make_hyper_samples, make_problem

ALL_KERNELS = [OB.KERNEL_SE, OB.KERNEL_MATERN32, OB.KERNEL_MATERN52, KERNEL_MATERN12, RQ(0.5), RQ(2.0), RQ(50.0)]
IDS = ["se", "matern32", "matern52", "matern12", "rq0.5", "rq2", "rq50"]


@pytest.mark.parametrize("kernel", ALL_KERNELS, ids=IDS)
def test_longdouble_gradient_matches_mpmath(kernel):
    pytest.importorskip("mpmath")
    n, d = 10, 3
    X, Y, _, _, _ = make_problem(n, d, seed=40)
    L, A, N = make_hyper_samples(2, d, seed=41)
    mask = np.array([False, True, False])
    Xd = X.copy(); Xd[1] = X[1] * 3                       # a discrete dimension with a few distinct levels
    for s, (Xs, m) in enumerate(((X, None), (Xd, mask))):
        ll, g = LS.adjudicator_grad_longdouble(Xs, Y[0], L[s], A[s], N[s], kernel, m)
        ll_mp, g_mp = LS.mp_loglik_grad(Xs, Y[0], L[s], A[s], N[s], kernel, m)
        assert abs(ll - ll_mp) <= 1e-15 * abs(ll_mp)
        assert np.max(np.abs(g - g_mp)) <= 1e-14 * np.linalg.norm(g_mp), (g, g_mp)
        if m is not None:
            assert g[1] != 0.0                              # a discrete dimension's lengthscale still scales K


@pytest.mark.parametrize("kernel", [OB.KERNEL_MATERN52, KERNEL_MATERN12, RQ(2.0)], ids=["matern52", "matern12", "rq2"])
def test_fp64_reference_is_far_inside_the_gradient_tolerance_at_n1024(kernel):
    """Justifies the FP64 oracle as the GPU tests' reference at eight blocks: its distance from the long-double truth,
    per sample, is printed and must be below 1e-10 |g| (a hundredth of the GPU tolerance)."""
    n, d = 1024, 8
    X, Y, _, _, _ = make_problem(n, d, seed=1024)
    L, A, N = make_hyper_samples(2, d, seed=1025)
    for s in range(2):
        ll_t, g_t = LS.adjudicator_grad_longdouble(X, Y[0], L[s], A[s], N[s], kernel)
        ll_o, g_o = LS.reference_grad(X, Y[0], L[s], A[s], N[s], kernel)
        e_g = float(np.max(np.abs(g_o - g_t)) / np.linalg.norm(g_t))
        e_l = abs(ll_o - ll_t) / abs(ll_t)
        print(f"n={n} {kernel} sample {s}: FP64 oracle vs long double: grad {e_g:.2e} |g|, loglik {e_l:.2e} rel")
        assert e_g <= 1e-10 and e_l <= 1e-12


# The shapes of tests/test_gpu_loglik_scale.py's reference comparisons, each with the kernel it runs there
SENS_SHAPES = [(2048, 8, OB.KERNEL_MATERN52, 2048), (769, 32, KERNEL_MATERN12, 801), (1000, 32, RQ(2.0), 1032),
               (2047, 32, OB.KERNEL_SE, 2079)]


@pytest.mark.parametrize("n,d,kernel,seed", SENS_SHAPES)
def test_gradient_check_rejects_a_missing_tile_and_a_wrong_lengthscale(n, d, kernel, seed):
    X, Y, _, _, _ = make_problem(n, d, seed=seed)
    L, A, N = make_hyper_samples(1, d, seed=seed + 1)
    ref, part = LS.tile_contributions(X, Y[0], L[0], A[0], N[0], kernel)
    base = LS.reference_grad(X, Y[0], L[0], A[0], N[0], kernel)[1]
    assert LS.grad_ratio(ref, base) <= 1e-3                  # the tile split is the reference's own sum
    nblk = part.shape[0]
    worst = np.inf
    for bi in range(nblk):
        for bj in range(nblk):
            if bi != bj:                                     # one off-diagonal tile of G left out
                worst = min(worst, LS.grad_ratio(ref - part[bi, bj], ref))
    print(f"n={n} d={d}: smallest miss / tolerance over {nblk * (nblk - 1)} dropped tiles: {worst:.3g}")
    assert worst > 1.0
    lows = []
    qs = range(d) if d <= 8 else (0, d // 2, d - 1)
    for q in qs:                                             # one lengthscale off by a relative 1e-5
        Lq = L[0].copy(); Lq[q] *= 1 + 1e-5
        lows.append(LS.grad_ratio(LS.reference_grad(X, Y[0], Lq, A[0], N[0], kernel)[1], ref))
    print(f"n={n} d={d}: smallest miss / tolerance over lengthscales {list(qs)} off by 1e-5: {min(lows):.3g}")
    assert min(lows) > 1.0


def test_window_plan_counts_windows():
    for mode in ("value", "grad", "fit"):
        Sb = LS.window_plan(100, 3, 10 ** 6, mode)["Sb"]
        assert Sb == 32768                                   # n_pad = 128: the 32768 cap, not the workspace, binds
        assert len(LS.window_plan(100, 3, Sb, mode)["windows"]) == 1
        p = LS.window_plan(100, 3, Sb + 1, mode)
        assert [(w["s0"], w["sb"]) for w in p["windows"]] == [(0, Sb), (Sb, 1)]
    p = LS.window_plan(4096, 4, 90, "grad")
    assert p["per"] == 411_041_792 and p["Sb"] == 83
    assert [w["groups"] for w in p["windows"]] == [[(0, 21), (21, 21), (42, 21), (63, 20)], [(83, 7)]]
    assert LS.window_plan(20, 2, 500, "value")["small"] and not LS.window_plan(20, 2, 500, "grad")["small"]


def test_window_plan_groups():
    (w,) = LS.window_plan(2048, 8, 10, "grad")["windows"]
    assert [g[1] for g in w["groups"]] == [3, 3, 3, 1]
    assert LS.boundary_samples(LS.window_plan(2048, 8, 10, "grad")) == [0, 2, 3, 5, 6, 8, 9]
    (w,) = LS.window_plan(900, 4, 37, "value", groups=16)["windows"]
    assert w["gsz"] == 3 and len(w["groups"]) == 13          # ceil(37 / 3) = 13: groups 13-15 are empty
    assert [g[1] for g in w["groups"]] == [3] * 12 + [1]
    for g, sizes in ((1, [37]), (2, [19, 18]), (3, [13, 13, 11]), (4, [10, 10, 10, 7]), (5, [8, 8, 8, 8, 5])):
        (w,) = LS.window_plan(900, 4, 37, "grad", groups=g)["windows"]
        assert [x[1] for x in w["groups"]] == sizes
    (w,) = LS.window_plan(900, 4, 37, "grad", groups=4, timing=True)["windows"]
    assert w["ngroups"] == 1
    (w,) = LS.window_plan(900, 4, 7, "grad")["windows"]      # fewer than 2 samples a group: one group
    assert w["ngroups"] == 1
    (w,) = LS.window_plan(300, 4, 8, "grad")["windows"]      # nblk <= 6: two groups by default
    assert w["ngroups"] == 2
    assert LS.window_plan(900, 4, 37, "value", groups=99)["windows"][0]["ngroups"] == 16
    assert LS.window_plan(900, 4, 37, "value", groups=0)["windows"][0]["ngroups"] == 1
