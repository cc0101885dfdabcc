#!/usr/bin/env python
"""Posterior x-gradients as an output (boss_gp_predict_grad, DESIGN.md 2.12) and the NonlinFitness closures
differentiated through them, alternated in one process.

  python tools/bench_predict_grad.py [--rounds 3] [--steps 5] [--out FILE]

(a) C4's shape (n = 4096, d = 4, Matern52, 1024 candidates), y_dim = 1 and 4: boss_gp_predict_grad against
    boss_ei_value_grad (same pipeline, acq_grad_kernel in place of the transposing output stage), ms per call, and a
    torch.profiler run of each: GPU time per kernel name, and predict_grad_kernel's share of the call's GPU time;
(b) 1 Mi candidates at n = 2048, d = 8, y_dim = 4 (28 chunks) from pageable and from pinned memory, ms per call and
    the output stage's share;
(c) the mirror's OptimizationAM on a two-output problem: a NonlinFitness closure with `grad` (host L-BFGS over
    boss_gp_predict_grad + the host chain rule) against the same fitness as an ExprFitness (the device multi-start
    driver), and one value + gradient pass over 1024 starts x 200 eps of each (host chain rule vs
    boss_mcei_value_grad).
One JSON line, with the card name and power limit it was measured at."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

from tools.bench_screen import card  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from torch.profiler import ProfilerActivity, profile
    import boss_b200 as B
    from boss_b200 import _lib
    from boss_b200 import acquisition_maximizers as AMs
    from boss_b200.acquisition import Acquisition
    from tests.util_problems import make_problem
    _lib.init(0)

    def timed(fn, steps):
        fn()                                     # warm-up (and this mode's scratch sizes)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(steps):
            r = fn()
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) / steps * 1e3, r

    def kernels(fn, steps):
        """GPU time per kernel name of one call (ms), from a profiler run of its own"""
        fn()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(steps):
                fn()
            torch.cuda.synchronize()
        per = {}
        for e in prof.key_averages():
            t = getattr(e, "device_time_total", None)
            t = e.cuda_time_total if t is None else t
            if t > 0:
                per[e.key] = t / steps / 1e3
        tot = sum(per.values())
        stage = sum(v for k, v in per.items() if "predict_grad_kernel" in k)
        acqg = sum(v for k, v in per.items() if "acq_grad_kernel" in k)
        return {"total_ms": tot, "predict_grad_kernel_ms": stage, "acq_grad_kernel_ms": acqg,
                "predict_grad_kernel_share": stage / tot if tot else None, "per_kernel_ms": per}

    def alternate(arms, steps):
        ms = {a: [] for a in arms}
        for _ in range(args.rounds):
            for a, fn in arms.items():
                ms[a].append(timed(fn, steps)[0])
        return ms, {a: float(np.median(v)) for a, v in ms.items()}

    out = {"card": card(), "rounds": args.rounds, "steps": args.steps}

    # ---- (a) C4's shape ----
    n, d, M = 4096, 4, 1024
    res = {}
    for y_dim in (1, 4):
        X, Y, ls, amp, ns = make_problem(n, d, seed=1004, y_dim=y_dim)
        gps = [_lib.gp_fit(X, Y[i], ls[i], amp[i], ns[i], _lib.KERNEL_MATERN52) for i in range(y_dim)]
        Xs = np.random.default_rng(1).random((d, M))
        co = np.full(y_dim, 1.0 / y_dim)
        best = float(np.median(co @ Y))
        arms = {"predict_grad": lambda: _lib.gp_predict_grad(gps, y_dim, 1, Xs),
                "ei_value_grad": lambda: _lib.ei_value_grad(gps, y_dim, 1, Xs, co, best, None)}
        ms, med = alternate(arms, args.steps)
        res[f"y_dim_{y_dim}"] = {"ms": ms, "median_ms": med, "predict_over_ei": med["predict_grad"] / med["ei_value_grad"],
                                 "gpu_time_per_call": {a: kernels(fn, args.steps) for a, fn in arms.items()}}
        for g in gps:
            g.free()
    out["a_c4_shape"] = {"n": n, "d": d, "M": M, **res}
    print("a", json.dumps(out["a_c4_shape"]), file=sys.stderr, flush=True)

    # ---- (b) 1 Mi candidates, pageable and pinned ----
    n, d, y_dim, M = 2048, 8, 4, 1 << 20
    X, Y, ls, amp, ns = make_problem(n, d, seed=1002, y_dim=y_dim)
    gps = [_lib.gp_fit(X, Y[i], ls[i], amp[i], ns[i], _lib.KERNEL_MATERN52) for i in range(y_dim)]
    Xs = np.random.default_rng(2).random((d, M))
    pinned = torch.empty((M, d), dtype=torch.float64, pin_memory=True)
    pinned.copy_(torch.from_numpy(np.ascontiguousarray(Xs.T)))
    Xp = pinned.numpy().T
    arms = {"pageable": lambda: _lib.gp_predict_grad(gps, y_dim, 1, Xs), "pinned": lambda: _lib.gp_predict_grad(gps, y_dim, 1, Xp)}
    ms, med = alternate(arms, 1)
    same = all(np.array_equal(a, b) for a, b in zip(arms["pageable"](), arms["pinned"]()))
    prof = kernels(arms["pinned"], 1)
    prof.pop("per_kernel_ms")
    out["b_1mi"] = {"n": n, "d": d, "y_dim": y_dim, "M": M, "chunks": -(-M // (296 * 128)), "ms": ms, "median_ms": med,
                    "M_candidates_per_s": {a: M / v / 1e3 for a, v in med.items()}, "pageable_equals_pinned": bool(same),
                    "gpu_time_pinned": prof}
    print("b", json.dumps(out["b_1mi"]), file=sys.stderr, flush=True)
    del pinned
    for g in gps:
        g.free()

    # ---- (c) the mirror: OptimizationAM on a closure with grad vs the ExprFitness device driver ----
    f = lambda x: np.array([np.sin(x[0]) + 0.1 * x[1], np.cos(x[0]) - 0.05 * x[1]])
    dom = B.Domain(([0.0, 0.0], [10.0, 10.0]))
    Xd = B.generate_LHC(dom.bounds, 20, np.random.default_rng(0))
    Yd = np.stack([f(Xd[:, j]) for j in range(20)], axis=1)
    model = B.GaussianProcess(kernel=B.SqExponentialKernel(), lengthscale_priors=[B.mvlognormal([0.5, 0.5], [0.5, 0.5])] * 2,
                              amplitude_priors=[B.LogNormal(0.0, 0.5)] * 2, noise_std_priors=[B.Dirac(0.1)] * 2)
    ex = B.ExprFitness("max", [1.0, 0.8], t=[0.0, 0.1])
    prob = B.BossProblem(f, dom, B.ExpectedImprovement(ex, eps_samples=200), model, B.ExperimentData(Xd, Yd))
    prob.params = B.estimate_parameters(B.SamplingMAP(64, seed=1), prob)
    post = B.model_posterior(prob)
    eps = np.random.default_rng(3).standard_normal((2, 200))
    best = B.best_so_far(prob, ex)

    def gmax(Z):      # df/dy of the max: the first extreme output's coefficient
        v = ex.c[:, None] * Z + ex.t[:, None]
        G = np.zeros_like(Z)
        pick = np.argmax(v, axis=0)
        G[0] = np.where(pick == 0, ex.c[0], 0.0)
        G[1] = np.where(pick == 1, ex.c[1], 0.0)
        return G

    acq_e = Acquisition(prob, post, prob.acquisition, best, eps)
    acq_c = Acquisition(prob, post, B.ExpectedImprovement(B.NonlinFitness(ex._eval, grad=gmax), eps_samples=200), best, eps)
    starts = B.generate_LHC(dom.bounds, 1024, np.random.default_rng(4))
    arms = {"closure_host_chain_rule": lambda: acq_c.value_and_grad(starts),
            "expr_device": lambda: acq_e.value_and_grad(starts)}
    ms, med = alternate(arms, args.steps)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        _lib.gp_predict_grad(acq_c.slices, 2, 1, starts)
    torch.cuda.synchronize()
    t_pg = (time.perf_counter() - t0) / args.steps * 1e3
    st256 = starts[:, :256]
    solve = {"closure_host_lbfgs": lambda: B.maximize_acquisition(AMs.OptimizationAM(st256, iters=40), prob, acq=acq_c),
             "expr_device_driver": lambda: B.maximize_acquisition(AMs.OptimizationAM(st256, iters=40), prob, acq=acq_e)}
    sms, smed = alternate(solve, 1)
    vals = {a: float(fn()[1]) for a, fn in solve.items()}
    out["c_mirror"] = {"y_dim": 2, "n": 20, "eps": 200, "pass_starts": 1024, "pass_ms": ms, "pass_median_ms": med,
                       "gp_predict_grad_part_ms": t_pg, "solve_starts": 256, "solve_iters": 40, "solve_ms": sms,
                       "solve_median_ms": smed, "solve_best_val": vals}
    print("c", json.dumps(out["c_mirror"]), file=sys.stderr, flush=True)
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f_:
            f_.write(line + "\n")


if __name__ == "__main__":
    main()
