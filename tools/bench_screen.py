#!/usr/bin/env python
"""Argmax screening (DESIGN.md 2.9) against the full path, alternated in one process.

  python tools/bench_screen.py [--rounds 3] [--steps 3] [--out FILE]

Cases: bench.py's problem (n = 2048, d = 8, Matern52, 2 Mi candidates) with the candidates resident on the device, in
pinned and in pageable host memory; C5's shape (n = 1024, d = 10, 4 outputs, EI x PoF, 512 Ki candidates, argmax only);
and the worst case for screening, 2 Mi identical candidates at the bench problem (every bound ties, the call falls back
after the first chunk).  Each round times `steps` screened calls, then `steps` calls with BOSS_NO_SCREEN=1; printed per
case: ms per call of both, the survivor fraction and whether the (value, index) pairs are bit-identical.  One JSON line,
with the card name and power limit it was measured at."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clk = [t.strip() for t in q.split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": clk}
    except Exception as e:  # noqa: BLE001
        return {"error": repr(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import boss_b200  # noqa: F401
    from boss_b200 import _lib
    from oracle import boss_oracle as O
    from tests.util_problems import make_problem
    _lib.init(0)

    X, Y, ls, amp, ns = make_problem(2048, 8, seed=1002)
    gp = _lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], _lib.KERNEL_MATERN52)
    best = float(np.max(Y[0]))
    M = 1 << 21
    gen = torch.Generator(device="cuda")
    gen.manual_seed(2002)
    Xs_dev = torch.rand((M, 8), dtype=torch.float64, device="cuda", generator=gen)     # bench.py's candidates
    Xs_pin = torch.empty((M, 8), dtype=torch.float64, pin_memory=True)
    Xs_pin.copy_(Xs_dev)
    Xs_pg = np.array(Xs_pin.numpy(), copy=True).T
    Xs_same = torch.full((M, 8), 0.37, dtype=torch.float64, device="cuda")

    n5, d5, y5, M5 = 1024, 10, 4, 1 << 19
    X5, Y5, ls5, amp5, ns5 = make_problem(n5, d5, seed=1005, y_dim=y5)
    gps5 = [_lib.gp_fit(X5, Y5[i], ls5[i], amp5[i], ns5[i], _lib.KERNEL_MATERN52) for i in range(y5)]
    y_max5 = np.array([np.inf] + [float(np.quantile(Y5[i], 0.7)) for i in range(1, y5)])
    coefs5 = np.array([1.0, 0, 0, 0])
    best5 = O.best_so_far(coefs5, Y5, y_max5)
    Xs5 = torch.rand((M5, d5), dtype=torch.float64, device="cuda", generator=gen)
    torch.cuda.synchronize()

    cases = {
        "bench_resident": (M, lambda: _lib.ei_score_dev([gp], 1, 1, Xs_dev.data_ptr(), M, [1.0], best, None)),
        "bench_e2e_pinned": (M, lambda: _lib.ei_score([gp], 1, 1, Xs_pin.numpy().T, [1.0], best, None, want_acq=False)[1:]),
        "bench_e2e_pageable": (M, lambda: _lib.ei_score([gp], 1, 1, Xs_pg, [1.0], best, None, want_acq=False)[1:]),
        "c5_shape_argmax": (M5, lambda: _lib.ei_score_dev(gps5, y5, 1, Xs5.data_ptr(), M5, coefs5, best5, y_max5)),
        "worst_identical": (M, lambda: _lib.ei_score_dev([gp], 1, 1, Xs_same.data_ptr(), M, [1.0], best, None)),
    }

    def timed(fn, steps):
        fn()                                     # warm-up (and this mode's scratch sizes)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(steps):
            r = fn()
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) / steps * 1e3, r

    out = {"card": card(), "rounds": args.rounds, "steps": args.steps, "cases": {}}
    for name, (m, fn) in cases.items():
        on, off, stats, same = [], [], None, True
        for _ in range(args.rounds):
            os.environ.pop("BOSS_NO_SCREEN", None)
            ms1, r1 = timed(fn, args.steps)
            stats = _lib.dbg_screen_stats()
            os.environ["BOSS_NO_SCREEN"] = "1"
            ms0, r0 = timed(fn, args.steps)
            os.environ.pop("BOSS_NO_SCREEN", None)
            on.append(ms1)
            off.append(ms0)
            same = same and (np.float64(r1[0]).view(np.int64) == np.float64(r0[0]).view(np.int64)) and r1[1] == r0[1]
        out["cases"][name] = {
            "M": m, "ms_screened": on, "ms_full": off, "speedup_median": float(np.median(off) / np.median(on)),
            "cand_per_s_screened_median": m / (np.median(on) * 1e-3), "cand_per_s_full_median": m / (np.median(off) * 1e-3),
            "screen_state": stats[0], "bounded": stats[1], "survivors": stats[2],
            "survivor_fraction": stats[2] / max(stats[1], 1), "pairs_bit_identical": bool(same)}
        print(name, json.dumps(out["cases"][name]), file=sys.stderr, flush=True)
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
