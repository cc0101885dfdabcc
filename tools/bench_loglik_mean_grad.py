#!/usr/bin/env python
"""The prior-mean theta-gradient of the log-likelihood (boss_gp_loglik_grad_batch_mean, DESIGN.md 2.13) against the
hyper-parameter gradient call it extends (boss_gp_loglik_grad_batch), alternated in one process on identical inputs.

  python tools/bench_loglik_mean_grad.py [--rounds 3] [--steps 3] [--out FILE]

(a) the headline log-likelihood shape, n = 2048, d = 8, S = 256, Matern52, k = 2 and 16, J shared (ldj = 0) and per
    sample, all from pageable host memory: ms per call, the extra ms over the hyper-parameter call, the GPU time of
    loglik_mean_grad_kernel from a torch.profiler run of its own, and the time of the per-sample J's host-to-device copy
    alone (S*n*k*8 bytes from the same pageable array); loglik and grad compared bit for bit;
(b) C4's shape, n = 4096, d = 4, k = 2, S = 32, shared and per-sample J, the same figures;
(c) the mirror's Semiparametric OptimizationMAP, "lbfgs" (on the new call) against "compass" (value-only batches), on
    y = 2 x_1 + 0.5 + residual at n = 200: wall time, library calls and the final log-likelihood.
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
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from torch.profiler import ProfilerActivity, profile
    import boss_b200 as B
    from boss_b200 import _lib
    from tests.util_problems import make_hyper_samples, make_problem
    _lib.init(0)

    def timed(fn, steps):
        fn()                                     # warm-up (and this mode's scratch sizes)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(steps):
            r = fn()
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) / steps * 1e3, r

    def alternate(arms, steps):
        ms = {a: [] for a in arms}
        for _ in range(args.rounds):
            for a, fn in arms.items():
                ms[a].append(timed(fn, steps)[0])
        return ms, {a: float(np.median(v)) for a, v in ms.items()}

    def kernel_ms(fn, steps):
        """GPU time of loglik_mean_grad_kernel and of all kernels of one call (ms), from a profiler run of its own"""
        fn()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(steps):
                fn()
            torch.cuda.synchronize()
        mg = tot = 0.0
        for e in prof.key_averages():
            t = getattr(e, "device_time_total", None)
            t = e.cuda_time_total if t is None else t
            tot += t
            if "loglik_mean_grad_kernel" in e.key:
                mg += t
        return {"loglik_mean_grad_kernel_ms": mg / steps / 1e3, "all_gpu_activity_ms": tot / steps / 1e3}

    def copy_ms(J, steps):
        """host-to-device copy of the per-sample J alone, from the same pageable array"""
        dst = torch.empty(J.shape, dtype=torch.float64, device="cuda")
        src = torch.from_numpy(J)
        dst.copy_(src)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(steps):
            dst.copy_(src)
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) / steps * 1e3

    def shape(n, d, S, ks, seed):
        X, Y, _, _, _ = make_problem(n, d, seed=seed)
        L, A, N = make_hyper_samples(S, d, seed=seed + 1)
        rng = np.random.default_rng(seed + 2)
        res = {}
        for k in ks:
            for per_sample in (False, True):
                J = rng.standard_normal((S, k, n) if per_sample else (k, n))
                Ymm = np.ascontiguousarray(Y[0] - 0.1 * rng.standard_normal((S, n)))    # per-sample delta, as the mirror
                arms = {"mean": lambda: _lib.loglik_grad_batch_mean(X, Ymm, J, L, A, N, _lib.KERNEL_MATERN52),
                        "hyper": lambda: _lib.loglik_grad_batch(X, Ymm, L, A, N, _lib.KERNEL_MATERN52)}
                ms, med = alternate(arms, args.steps)
                a, b = arms["mean"](), arms["hyper"]()
                same = bool(np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]))
                key = f"k{k}_{'per_sample' if per_sample else 'shared'}"
                res[key] = {"ms": ms, "median_ms": med, "extra_ms": med["mean"] - med["hyper"],
                            "extra_fraction": med["mean"] / med["hyper"] - 1.0, "loglik_grad_bit_identical": same,
                            "J_bytes": int(J.nbytes), "gpu_time": kernel_ms(arms["mean"], 1),
                            "J_copy_alone_ms": copy_ms(J, args.steps) if per_sample else 0.0}
                print(key, json.dumps(res[key]), file=sys.stderr, flush=True)
        return {"n": n, "d": d, "S": S, "kernel": "Matern52", "source": "pageable", **res}

    out = {"card": card(), "rounds": args.rounds, "steps": args.steps}
    out["a_headline"] = shape(2048, 8, 256, (2, 16), seed=2048)
    out["b_c4_shape"] = shape(4096, 4, 32, (2,), seed=4096)

    # ---- (c) the mirror: Semiparametric OptimizationMAP, gradient vs compass ----
    from tests.test_loglik_mean_grad_host import linear_problem
    prob = linear_problem(B, n=200)
    counts = {"loglik_batch": 0, "loglik_grad_batch_mean": 0}
    for name in counts:
        f0 = getattr(_lib, name)

        def wrapped(*a, _f=f0, _n=name, **kw):
            counts[_n] += 1
            return _f(*a, **kw)
        setattr(_lib, name, wrapped)
    res = {}
    for alg in ("lbfgs", "compass"):
        for c in counts:
            counts[c] = 0
        t0 = time.perf_counter()
        r = B.estimate_parameters(B.OptimizationMAP(multistart=12, iters=30, seed=21, algorithm=alg), prob)
        res[alg] = {"wall_s": time.perf_counter() - t0, "library_calls": dict(counts), "loglike": r.loglike,
                    "theta": [float(t) for t in r.params.theta]}
    out["c_mirror"] = {"n": 200, "multistart": 12, "iters": 30, **res}
    print("c", json.dumps(out["c_mirror"]), file=sys.stderr, flush=True)
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f_:
            f_.write(line + "\n")


if __name__ == "__main__":
    main()
