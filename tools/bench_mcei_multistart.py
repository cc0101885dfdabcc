#!/usr/bin/env python
"""OptimizationAM / SampleOptAM on the Monte-Carlo EI of an expression fitness (boss_mcei_value_grad,
boss_mcei_maximize_multistart, boss_mcei_score_topk; DESIGN.md 2.11) against their LinFitness twins, alternated in one
process.

  python tools/bench_mcei_multistart.py [--rounds 3] [--steps 5] [--out FILE]

(a) one value + gradient pass over 1024 starts at C4's shape (n = 4096, d = 4, one output, Matern52, K = 200 eps
    columns): boss_ei_value_grad against boss_mcei_value_grad of each of the four kinds, ms per pass, and a
    torch.profiler run of the LinFitness and max passes: GPU time per kernel name;
(b) the whole 50-iteration multi-start solve over those 1024 starts: boss_ei_maximize_multistart against
    boss_mcei_maximize_multistart (kind 1 with f(y) = y, the LinFitness objective), and once the host twin
    (batched_lbfgs_maximize over mcei_value_grad).
    In (a) and (b) every arm's `best` is the median of its fitness over the training outputs;
(c) C5's shape (n = 1024, d = 10, y_dim = 4, kind 3 "max"), 512 Ki candidates, k = 64: boss_mcei_score_topk against
    boss_mcei_score with every score to the host and a host julia_sortperm_rev.
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
    import boss_b200 as B
    from boss_b200 import _lib
    from boss_b200.acquisition import julia_sortperm_rev
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

    out = {"card": card(), "rounds": args.rounds, "steps": args.steps}

    # ---- (a) + (b): C4's shape ----
    n, d, S0, K = 4096, 4, 1024, 200
    X, Y, ls, amp, ns = make_problem(n, d, seed=1004)
    gp = _lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], _lib.KERNEL_MATERN52)
    best = float(np.median(Y[0]))
    lb, ub = np.zeros(d), np.ones(d)
    starts = B.generate_LHC((lb, ub), S0, np.random.default_rng(1))
    eps = np.random.default_rng(2).standard_normal((1, K))
    expr = {1: dict(c0=0.0, c=[1.0]), 2: dict(c0=0.1, c=[1.0], q=[-0.3], t=[0.1]), 3: dict(c=[1.0], t=[0.1]),
            4: dict(c=[-1.0], t=[0.1])}
    fit = {1: Y[0], 2: 0.1 + Y[0] - 0.3 * (Y[0] - 0.1) ** 2, 3: Y[0] + 0.1, 4: 0.1 - Y[0]}
    bests = {k: float(np.median(v)) for k, v in fit.items()}
    arms = {"lin": lambda: _lib.ei_value_grad([gp], 1, 1, starts, [1.0], best, None, lb, ub)}
    for kind, kw in expr.items():
        arms[f"mc_kind{kind}"] = (lambda kind=kind, kw=kw:
                                  _lib.mcei_value_grad([gp], 1, 1, starts, kind, eps, bests[kind], None, lb=lb, ub=ub, **kw))
    ms = {a: [] for a in arms}
    nonzero = {}
    for _ in range(args.rounds):
        for a, fn in arms.items():
            t, r = timed(fn, args.steps)
            ms[a].append(t)
            nonzero[a] = float(np.mean(np.any(r[1] != 0, axis=0)))
    med = {a: float(np.median(v)) for a, v in ms.items()}
    out["a_value_grad_pass"] = {"n": n, "d": d, "starts": S0, "eps": K, "ms": ms, "median_ms": med,
                                "mc_over_lin": {a: med[a] / med["lin"] for a in med if a != "lin"},
                                "share_of_starts_with_nonzero_gradient": nonzero}
    # where the difference goes: GPU time per kernel of one pass (profiler in its own loop, after the timed rounds)
    from torch.profiler import ProfilerActivity, profile
    kern = {}
    for a in ("lin", "mc_kind3"):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(args.steps):
                arms[a]()
            torch.cuda.synchronize()
        per = {}
        for e in prof.key_averages():
            t = getattr(e, "device_time_total", None)
            t = e.cuda_time_total if t is None else t
            if t > 0:
                per[e.key] = t / args.steps / 1e3      # ms per pass
        kern[a] = {"total_ms": sum(per.values()), "per_kernel_ms": per}
    out["a_value_grad_pass"]["gpu_time_per_pass"] = kern
    print("a", json.dumps(out["a_value_grad_pass"]), file=sys.stderr, flush=True)

    kw1 = expr[1]
    solve = {"lin": lambda: _lib.ei_maximize_multistart([gp], 1, 1, starts, [1.0], best, None, lb, ub, iters=50),
             "mc_kind1": lambda: _lib.mcei_maximize_multistart([gp], 1, 1, starts, 1, eps, best, None, lb, ub, iters=50, **kw1)}
    ms = {a: [] for a in solve}
    res = {}
    for _ in range(args.rounds):
        for a, fn in solve.items():
            t, r = timed(fn, 1)
            ms[a].append(t)
            res[a] = {"best_val": r[3], "evals": r[5]}
    vg = lambda Z: _lib.mcei_value_grad([gp], 1, 1, Z, 1, eps, best, None, lb=lb, ub=ub, **kw1)
    t0 = time.perf_counter()
    _, fh = B.batched_lbfgs_maximize(vg, starts, lb, ub, iters=50)
    t_host = (time.perf_counter() - t0) * 1e3
    out["b_multistart_50_iters"] = {"starts": S0, "ms": ms, "median_ms": {a: float(np.median(v)) for a, v in ms.items()},
                                    "results": res, "host_twin_mc_kind1_ms": t_host,
                                    "host_twin_best_val": float(np.max(fh))}
    print("b", json.dumps(out["b_multistart_50_iters"]), file=sys.stderr, flush=True)
    gp.free()

    # ---- (c): C5's shape, top-k ----
    n5, d5, y5, M5, k5 = 1024, 10, 4, 512 * 1024, 64
    X, Y, ls, amp, ns = make_problem(n5, d5, seed=1005, y_dim=y5)
    gps = [_lib.gp_fit(X, Y[i], ls[i], amp[i], ns[i], _lib.KERNEL_MATERN52) for i in range(y5)]
    Xs = np.random.default_rng(3).random((d5, M5))
    eps5 = np.random.default_rng(4).standard_normal((y5, K))
    kw3 = dict(c=[1.0, 0.8, 0.0, 0.5], t=[0.0, 0.1, 0.0, -0.1])
    best5 = float(np.quantile(np.max(Y[[0, 1, 3]], axis=0), 0.9))

    def host():
        acq, _, _ = _lib.mcei_score(gps, y5, 1, Xs, 3, eps5, best5, None, **kw3)
        top = julia_sortperm_rev(acq)[:k5]
        return acq[top], top

    topk = {"host": host, "device": lambda: _lib.mcei_score_topk(gps, y5, 1, Xs, 3, eps5, best5, None, k5, **kw3)}
    ms = {a: [] for a in topk}
    same = True
    for _ in range(args.rounds):
        t, ra = timed(topk["host"], 1)
        ms["host"].append(t)
        t, rb = timed(topk["device"], 1)
        ms["device"].append(t)
        same = same and np.array_equal(ra[1], rb[1]) and np.array_equal(ra[0].view(np.int64), rb[0].view(np.int64))
    med = {a: float(np.median(v)) for a, v in ms.items()}
    out["c_topk"] = {"n": n5, "d": d5, "y_dim": y5, "M": M5, "k": k5, "eps": K, "ms": ms, "median_ms": med,
                     "speedup_device_vs_host": med["host"] / med["device"], "results_identical": bool(same)}
    print("c", json.dumps(out["c_topk"]), file=sys.stderr, flush=True)
    for g in gps:
        g.free()
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
