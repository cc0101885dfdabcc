#!/usr/bin/env python
"""The five covariance functions side by side at the headline shape (n = 2048, d = 8), alternated in one process:
SqExponential, Matern32, Matern52, Matern12 (ExponentialKernel) and RationalQuadratic (a = 2).

  python tools/bench_kernels.py [--rounds 3] [--steps 5] [--out FILE]

Per kernel and round, after one warm-up call of each shape, the median over --steps synchronised calls of
  fit_ms          boss_gp_fit (host inputs)
  loglik_per_s    boss_gp_loglik_batch, S = 256 samples
  loglik_grad_per_s   boss_gp_loglik_grad_batch, S = 256
  argmax_ms       screened EI argmax over 2 Mi device-resident candidates (boss_ei_score_dev)
  full_cand_per_s the same call with BOSS_NO_SCREEN=1 (every candidate scored)
  value_grad_ms   one boss_ei_value_grad pass over 1024 starts
and the screened / full pairs compared.  The reported figure is the median over rounds, with the min-max spread.
One JSON line, with the card name, power limit and max SM clock read in the same run."""
import argparse
import json
import os
import statistics
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

from tools.bench_screen import card  # noqa: E402

N, D, S, M, STARTS = 2048, 8, 256, 2 * 1024 * 1024, 1024


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from boss_b200 import _lib
    from tests.util_problems import make_hyper_samples, make_problem

    _lib.init(0)
    kernels = {"se": _lib.KERNEL_SE, "matern32": _lib.KERNEL_MATERN32, "matern52": _lib.KERNEL_MATERN52,
               "matern12": _lib.KERNEL_MATERN12, "rq2": _lib.kernel_rational_quadratic(2.0)}
    X, Y, ls, amp, ns = make_problem(N, D, seed=1)
    L, A, Nn = make_hyper_samples(S, D, seed=3)
    best = float(np.max(Y[0]))
    g = torch.Generator(device="cuda").manual_seed(2)
    xs = torch.rand((M, D), dtype=torch.float64, device="cuda", generator=g)   # column-major d x M
    starts = np.random.default_rng(4).random((D, STARTS))
    torch.cuda.synchronize()

    def timed(fn):
        fn()
        ts = []
        for _ in range(args.steps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            ts.append(time.perf_counter() - t0)
        return statistics.median(ts)

    def argmax(gp):
        return _lib.ei_score_dev([gp], 1, 1, xs.data_ptr(), M, [1.0], best, None)

    rounds = {k: [] for k in kernels}
    pairs_equal = {}
    for _ in range(args.rounds):
        for name, kid in kernels.items():
            r = {}
            r["fit_ms"] = 1e3 * timed(lambda: _lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], kid).free())
            r["loglik_per_s"] = S / timed(lambda: _lib.loglik_batch(X, Y[0], L, A, Nn, kid))
            r["loglik_grad_per_s"] = S / timed(lambda: _lib.loglik_grad_batch(X, Y[0], L, A, Nn, kid))
            gp = _lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], kid)
            r["argmax_ms"] = 1e3 * timed(lambda: argmax(gp))
            pair = argmax(gp)
            r["screened"] = _lib.dbg_screen_stats()[0]
            r["ambiguous"] = _lib.dbg_screen_ambiguous()[0]
            os.environ["BOSS_NO_SCREEN"] = "1"
            r["full_cand_per_s"] = M / timed(lambda: argmax(gp))
            full = argmax(gp)
            del os.environ["BOSS_NO_SCREEN"]
            pairs_equal[name] = pairs_equal.get(name, True) and pair == full
            r["value_grad_ms"] = 1e3 * timed(lambda: _lib.ei_value_grad([gp], 1, 1, starts, [1.0], best, None))
            gp.free()
            rounds[name].append(r)

    out = {"what": "five covariance functions at n = 2048, d = 8 (tools/bench_kernels.py)", "card": card(),
           "rounds": args.rounds, "steps": args.steps, "S": S, "M": M, "starts": STARTS,
           "screened_pair_equals_full": pairs_equal, "kernels": {}}
    for name, rs in rounds.items():
        agg = {}
        for key in rs[0]:
            vals = [r[key] for r in rs]
            if key in ("screened", "ambiguous"):
                agg[key] = vals[-1]
            else:
                agg[key] = {"median": statistics.median(vals), "min": min(vals), "max": max(vals)}
        out["kernels"][name] = agg
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")
    _lib.shutdown()


if __name__ == "__main__":
    main()
