#!/usr/bin/env python
"""One small call through every kernel family of libboss_b200.so, for compute-sanitizer (SURVEY.md 5 row 2):

    compute-sanitizer --tool memcheck  --error-exitcode 1 python tools/sanitizer_subset.py
    compute-sanitizer --tool racecheck --error-exitcode 1 python tools/sanitizer_subset.py --tiny

Families: build_k, potrf_tile (+ fused diagonal step), chol_trsm, chol_update, chol_panel, chol_update_rl, trtri_*_rl,
trtri_fused, kinv_wtw, loglik_grad_tile, loglik_mean_grad, loglik_small (warp path), matvec, xcov, score_trmm (plain and row-split),
wtv, grad (+ MC-EI gradient, + posterior gradients), acq (+ MC-EI), argmax, top-k, cov (gemm_nt + cov_finish), candidate generators, append (+ capacity growth),
multi-start driver.  Results are checked against the oracle so that a run that "passes" the sanitizer by computing
nothing is caught.  Prints one JSON line.
"""
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    tiny = "--tiny" in sys.argv
    import boss_b200  # noqa: F401
    from boss_b200 import _lib
    from oracle import boss_oracle as O
    from tests.util_problems import make_hyper_samples, make_problem, relerr
    t0 = time.time()
    _lib.init(0)
    done = []
    n, d = (200, 3) if tiny else (300, 4)          # 2 resp. 3 diagonal blocks: every block-column kernel runs
    X, Y, ls, amp, ns = make_problem(n, d, seed=1, y_dim=2)
    # --- fit (right-looking single-matrix path) + predict + EI (plain) ---
    gps = [_lib.gp_fit(X, Y[i], ls[i], amp[i], ns[i], 2 if i == 0 else 1) for i in range(2)]
    posts = [O.posterior_fit(X, Y[i], ls[i], amp[i], ns[i], 2 if i == 0 else 1) for i in range(2)]
    M = 300 if tiny else 1500
    rng = np.random.default_rng(2)
    Xs = rng.random((d, M))
    mu, var, st = _lib.gp_predict(gps[0], Xs)
    mo, vo, _ = O.mean_and_var(posts[0], Xs)
    assert relerr(var, vo) <= 1e-9 and np.max(np.abs(mu - mo)) <= 1e-9 * np.max(np.abs(mo))
    done.append("fit+predict")
    y_max = np.array([np.inf, float(np.quantile(Y[1], 0.7))])
    coefs = np.array([1.0, 0.0])
    best = O.best_so_far(coefs, Y, y_max)
    lb, ub = np.zeros(d), np.ones(d)
    acq, bv, bi = _lib.ei_score(gps, 2, 1, Xs, coefs, best, y_max, lb=lb, ub=ub)
    ref, _, _ = O.ei_acquisition([posts], Xs, coefs, best, y_max, lb=lb, ub=ub)
    m = ref > 1e-30 * ref.max()
    assert relerr(acq[m], ref[m]) <= 1e-9 and bi == O.julia_argmax_fast(ref)
    done.append("ei_score")
    # --- value + gradient (row-split trmm / wtv / grad / acq_grad) ---
    a_g, g_g = _lib.ei_value_grad(gps, 2, 1, Xs[:, :200], coefs, best, y_max, lb=lb, ub=ub)
    a_r, g_r = O.ei_value_grad(posts, Xs[:, :200], coefs, best, y_max)
    mm = a_r > 1e-30 * a_r.max()
    assert relerr(a_g[mm], a_r[mm]) <= 1e-9
    assert np.max(np.abs(g_g[:, mm] - g_r[:, mm]) / np.max(np.abs(g_r[:, mm]), axis=0)) <= 1e-7
    done.append("value_grad")
    # --- posterior x-gradients (predict_grad_kernel) for both slices in one call ---
    pmu, pvar, pdm, pdv, pst = _lib.gp_predict_grad(gps, 2, 1, Xs[:, :200])
    for i in range(2):
        mo, vo, dmo, dvo, _ = O.mean_var_grad(posts[i], Xs[:, :200])
        assert relerr(pvar[i], vo) <= 1e-9 and np.max(np.abs(pmu[i] - mo)) <= 1e-9 * np.max(np.abs(mo))
        assert np.max(np.abs(pdm[i] - dmo)) <= 1e-8 * np.max(np.abs(dmo))
        assert np.max(np.abs(pdv[i] - dvo)) <= 1e-8 * np.max(np.abs(dvo))
    done.append("predict_grad")
    # --- device candidate generators ---
    _, gv, gi, gx = _lib.ei_score_uniform(gps, 2, 1, 5, M, lb, ub, coefs, best, y_max)
    pts = _lib.uniform_candidates(5, 0, M, lb, ub)
    a_u, _, bi_u = _lib.ei_score(gps, 2, 1, pts, coefs, best, y_max, lb=lb, ub=ub)
    assert gi == bi_u
    cnt = np.array([6] * d)
    _, _, ggi, _ = _lib.ei_score_grid(gps, 2, 1, np.zeros(d), np.full(d, 0.2), cnt, coefs, best, y_max)
    assert 0 <= ggi < int(np.prod(cnt))
    done.append("generators")
    # --- MC-EI ---
    eps = rng.standard_normal((2, 16))
    a_mc, _, _ = _lib.mcei_score(gps, 2, 1, Xs[:, :256], 2, eps, best, y_max, c=coefs, q=np.array([0.0, -0.3]), t=np.zeros(2))
    f = lambda y: float(coefs @ y) - 0.3 * y[1] ** 2
    r_mc = O.mc_ei_acquisition([posts], Xs[:, :256], f, eps, best, y_max)
    assert np.max(np.abs(a_mc - r_mc)) <= 1e-9 * np.max(np.abs(r_mc))
    done.append("mcei")
    # --- MC-EI value + gradient, its multi-start driver and top-k (acq_grad_kernel<true>) ---
    from tests import mcei_grad_oracle as MO
    mc_kw = dict(c=coefs, q=np.array([0.0, -0.3]), t=np.zeros(2))
    best_mc = float(np.median([f(Y[:, j]) for j in range(n)]))      # most candidates improve on it: a non-trivial gradient
    a_mg, g_mg = _lib.mcei_value_grad(gps, 2, 1, Xs[:, :200], 2, eps, best_mc, y_max, **mc_kw)
    a_mr, g_mr = MO.mc_ei_value_grad([posts], Xs[:, :200], 2, 0.0, coefs, mc_kw["q"], mc_kw["t"], eps, best_mc, y_max)
    g_scale = np.max(np.abs(g_mr), axis=1, keepdims=True)
    assert np.all(g_scale > 0)
    assert np.max(np.abs(a_mg - a_mr)) <= 1e-9 * np.max(np.abs(a_mr))
    assert np.max(np.abs(g_mg - g_mr) / g_scale) <= 1e-7
    ms_starts = rng.random((d, 64))
    _, fo_mc, _, _, _, _ = _lib.mcei_maximize_multistart(gps, 2, 1, ms_starts, 2, eps, best_mc, y_max, lb, ub, iters=4,
                                                         **mc_kw)
    f0_mc, _, _ = _lib.mcei_score(gps, 2, 1, ms_starts, 2, eps, best_mc, y_max, lb=lb, ub=ub, **mc_kw)
    assert np.all(fo_mc >= f0_mc - 1e-15) and np.max(fo_mc) > 0
    a_tk, _, _ = _lib.mcei_score(gps, 2, 1, Xs[:, :256], 2, eps, best_mc, y_max, **mc_kw)
    tv_mc, ti_mc = _lib.mcei_score_topk(gps, 2, 1, Xs[:, :256], 2, eps, best_mc, y_max, 10, **mc_kw)
    assert np.array_equal(ti_mc, np.argsort(-a_tk, kind="stable")[:10]) and np.array_equal(tv_mc, a_tk[ti_mc])
    done.append("mcei_grad+multistart+topk")
    # --- full covariance ---
    mu_c, cov, _ = _lib.gp_cov(gps[0], Xs[:, :40])
    cref, _ = O.posterior_cov(posts[0], Xs[:, :40])
    assert np.max(np.abs(cov - cref)) <= 1e-9 * np.max(np.abs(cref))
    done.append("cov")
    # --- batched log-likelihood (left-looking batch path), + gradient (trtri_fused, kinv, grad tiles), + batch fit ---
    S = 6 if tiny else 20
    L, A, N = make_hyper_samples(S, d, seed=3)
    ll = _lib.loglik_batch(X, Y[0], L, A, N, 2)
    ll_ref = O.gp_loglik_batch(X, Y[0], L, A, N, 2)
    assert relerr(ll, ll_ref) <= 1e-8
    llg, gr = _lib.loglik_grad_batch(X, Y[0], L, A, N, 0)
    llr, grr = O.gp_loglik_grad_batch(X, Y[0], L, A, N, 0)
    assert relerr(llg, llr) <= 1e-8
    assert np.max(np.abs(gr - grr) / np.linalg.norm(grr, axis=1, keepdims=True)) <= 1e-8
    # prior-mean gradient (loglik_mean_grad_kernel), per-sample Jacobians: loglik and grad unchanged, alpha^T J
    from tests import loglik_mean_grad_oracle as MG
    Jm = np.random.default_rng(8).standard_normal((S, 3, n))
    llm, grm, gmm = _lib.loglik_grad_batch_mean(X, Y[0], Jm, L, A, N, 0)
    assert np.array_equal(llm, llg) and np.array_equal(grm, gr)
    _, gmr = MG.gp_loglik_mean_grad_batch(X, Y[0], Jm, L, A, N, 0)
    assert np.max(np.abs(gmm - gmr) / np.linalg.norm(gmr, axis=1, keepdims=True)) <= 1e-9
    fb = _lib.gp_fit_batch(X, Y[0], L[:3], A[:3], N[:3], 2)
    assert all(g is not None for g in fb)
    done.append("loglik+grad+mean_grad+fit_batch")
    # --- warp-register small-n path ---
    Xsm, Ysm, _, _, _ = make_problem(24, 2, seed=4)
    Ls, As, Ns = make_hyper_samples(40, 2, seed=5)
    lls = _lib.loglik_batch(Xsm, Ysm[0], Ls, As, Ns, 1)
    assert relerr(lls, O.gp_loglik_batch(Xsm, Ysm[0], Ls, As, Ns, 1)) <= 1e-8
    done.append("loglik_small")
    # --- append across a capacity boundary (n = 255 -> 257) ---
    Xa, Ya, la, aa, na = make_problem(255, 3, seed=6)
    ga = _lib.gp_fit(Xa, Ya[0], la[0], aa[0], na[0], 2)
    xn = np.random.default_rng(7).random((3, 2))
    for k in range(2):
        assert _lib.gp_append(ga, xn[:, k], 0.1 * k)
    Xfull = np.concatenate([Xa, xn], axis=1); yfull = np.concatenate([Ya[0], [0.0, 0.1]])
    pa = O.posterior_fit(Xfull, yfull, la[0], aa[0], na[0], 2)
    mu_a, var_a, _ = _lib.gp_predict(ga, Xs[:3, :100])
    mo_a, vo_a, _ = O.mean_and_var(pa, Xs[:3, :100])
    assert relerr(var_a, vo_a) <= 1e-8 and np.max(np.abs(mu_a - mo_a)) <= 1e-8 * np.max(np.abs(mo_a))
    done.append("append")
    # --- multi-start driver ---
    starts = rng.random((d, 64 if tiny else 200))
    Xo, fo, bx, bvm, bim, ev = _lib.ei_maximize_multistart(gps, 2, 1, starts, coefs, best, y_max, lb, ub, iters=4 if tiny else 8)
    f0, _, _ = _lib.ei_score(gps, 2, 1, starts, coefs, best, y_max, lb=lb, ub=ub)
    assert np.all(fo >= f0 - 1e-15)
    done.append("multistart")
    # guard bands of every live device allocation (BOSS_DEBUG_REDZONE=1): the workspaces are still alive here
    bad, nalloc = _lib.dbg_check_redzones()
    assert bad <= 0, f"{bad} guard bytes overwritten"
    selftest = int(_lib.lib.boss_dbg_redzone_selftest())      # negative control: 2 when the mode is on, -1 when off
    assert selftest in (2, -1), selftest
    for g in gps + fb + [ga]:
        g.free()
    nl = _lib.launch_count()
    _lib.shutdown()
    print(json.dumps({"sanitizer_subset": "ok", "tiny": tiny, "families": done, "launches": int(nl),
                      "redzone_bytes_overwritten": bad, "redzone_allocations_scanned": nalloc, "redzone_selftest_detected": selftest,
                      "seconds": time.time() - t0}))


if __name__ == "__main__":
    main()
