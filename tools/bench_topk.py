#!/usr/bin/env python
"""SampleOptAM's start selection: the device top-k (boss_ei_score_topk, DESIGN.md 2.10) against the host path it
replaces, alternated in one process.

  python tools/bench_topk.py [--rounds 3] [--steps 2] [--out FILE]

Problem: bench.py's (n = 2048, d = 8, Matern52), 2 Mi candidates in pageable host memory, as the sampler leaves them.
For each k in {1, 64, 1024, 8192} a round times, in turn, `steps` calls of
  (a) host:      every score to the host (boss_ei_score with the M-vector), then np.argsort(-vals, kind="stable")[:k]
  (b) screened:  boss_ei_score_topk
  (c) full:      boss_ei_score_topk with BOSS_NO_SCREEN=1.
Printed per k: ms per call of each, the screening state and survivor count of (b), and whether the three index lists
(and the values of (b) and (c), bit for bit) agree.  Only the selection is timed, not the sampler that draws the
candidates.  One JSON line, with the card name and power limit it was measured at."""
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
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import boss_b200  # noqa: F401
    from boss_b200 import _lib
    from tests.util_problems import make_problem
    _lib.init(0)

    X, Y, ls, amp, ns = make_problem(2048, 8, seed=1002)
    gp = _lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], _lib.KERNEL_MATERN52)
    best = float(np.max(Y[0]))
    M = 1 << 21
    Xs = np.random.default_rng(2002).random((8, M))

    def host(k):
        acq, _, _ = _lib.ei_score([gp], 1, 1, Xs, [1.0], best, None, want_acq=True)
        top = np.argsort(-acq, kind="stable")[:k]
        return acq[top], top

    def device(k):
        return _lib.ei_score_topk([gp], 1, 1, Xs, [1.0], best, None, k)

    def timed(fn, k, steps):
        fn(k)                                    # warm-up (and this mode's scratch sizes)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(steps):
            r = fn(k)
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) / steps * 1e3, r

    out = {"card": card(), "n": 2048, "d": 8, "M": M, "rounds": args.rounds, "steps": args.steps, "k": {}}
    for k in (1, 64, 1024, 8192):
        ms = {"host": [], "screened": [], "full": []}
        same, stats = True, None
        for _ in range(args.rounds):
            os.environ.pop("BOSS_NO_SCREEN", None)
            t, ra = timed(host, k, args.steps)
            ms["host"].append(t)
            t, rb = timed(device, k, args.steps)
            stats = _lib.dbg_screen_stats()
            ms["screened"].append(t)
            os.environ["BOSS_NO_SCREEN"] = "1"
            t, rc = timed(device, k, args.steps)
            os.environ.pop("BOSS_NO_SCREEN", None)
            ms["full"].append(t)
            same = same and np.array_equal(ra[1], rb[1]) and np.array_equal(rb[1], rc[1]) and \
                np.array_equal(rb[0].view(np.int64), rc[0].view(np.int64))
        med = {m: float(np.median(v)) for m, v in ms.items()}
        out["k"][str(k)] = {
            "ms_host": ms["host"], "ms_screened": ms["screened"], "ms_full": ms["full"], "median_ms": med,
            "speedup_screened_vs_host": med["host"] / med["screened"], "speedup_full_vs_host": med["host"] / med["full"],
            "screen_state": stats[0], "bounded": stats[1], "survivors": stats[2], "results_identical": bool(same)}
        print(k, json.dumps(out["k"][str(k)]), file=sys.stderr, flush=True)
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
