#!/usr/bin/env python
"""The FP32 mean tier of argmax screening alone (DESIGN.md 2.9): the CUDA time of its kernels in one device-resident
screened call, without re-seed, under torch.profiler (CUDA events inside the profiler's trace).

  python tools/bench_mean_tier.py [--calls 5] [--out FILE]

Cases: bench.py's problem (n = 2048, d = 8, Matern52, 2 Mi candidates) and C5's shape (n = 1024, d = 10, 4 outputs,
EI x PoF, 512 Ki candidates).  The tier's kernels are screen_mean_bound_kernel (means, bounds and survivor counts of
every candidate after the first chunk); older builds named them xcov_mean_mma_kernel and screen_tail_kernel, and those
are summed the same way, so the tool compares builds.  Printed per case: microseconds per call, (candidate, training
point) pairs per second per slice, and two bounds whose rates are assumptions, not measurements.  One JSON line with the
card name and power limit it was measured at."""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True
from tools.bench_screen_tiers import SASS_INSTR_PER_PAIR, card  # noqa: E402

TIER_KERNELS = ("screen_mean_bound_kernel", "xcov_mean_mma_kernel", "screen_tail_kernel")
SM_CLOCK = 1.965e9   # the card's maximum SM clock (sm_max_clock), for the assumed bounds


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from torch.profiler import ProfilerActivity, profile
    import boss_b200  # noqa: F401
    from boss_b200 import _lib
    from oracle import boss_oracle as O
    from tests.util_problems import make_problem
    _lib.init(0)
    os.environ.pop("BOSS_SCREEN_F64", None)
    os.environ["BOSS_SCREEN_NO_RESEED"] = "1"
    gen = torch.Generator(device="cuda")
    gen.manual_seed(2002)

    X, Y, ls, amp, ns = make_problem(2048, 8, seed=1002)
    gp = _lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], _lib.KERNEL_MATERN52)
    M = 1 << 21
    Xs = torch.rand((M, 8), dtype=torch.float64, device="cuda", generator=gen)
    n5, d5, y5, M5 = 1024, 10, 4, 1 << 19
    X5, Y5, ls5, amp5, ns5 = make_problem(n5, d5, seed=1005, y_dim=y5)
    gps5 = [_lib.gp_fit(X5, Y5[i], ls5[i], amp5[i], ns5[i], _lib.KERNEL_MATERN52) for i in range(y5)]
    y_max5 = np.array([np.inf] + [float(np.quantile(Y5[i], 0.7)) for i in range(1, y5)])
    coefs5 = np.array([1.0, 0, 0, 0])
    best5 = O.best_so_far(coefs5, Y5, y_max5)
    Xs5 = torch.rand((M5, d5), dtype=torch.float64, device="cuda", generator=gen)
    torch.cuda.synchronize()
    # (call, candidates, n_pad, slices); the first chunk (FP64 tier) is 592 blocks of 128 candidates at both shapes
    cases = {
        "bench": (lambda: _lib.ei_score_dev([gp], 1, 1, Xs.data_ptr(), M, [1.0], float(np.max(Y[0])), None), M, 2048, 1),
        "c5": (lambda: _lib.ei_score_dev(gps5, y5, 1, Xs5.data_ptr(), M5, coefs5, best5, y_max5), M5, 1024, y5),
    }
    out = {"card": card(), "calls": args.calls, "cases": {}}
    for name, (fn, m, n_pad, nsl) in cases.items():
        fn()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as pr:
            for _ in range(args.calls):
                fn()
            torch.cuda.synchronize()
        st = _lib.dbg_screen_stats()
        us, launches = 0.0, 0
        for e in pr.key_averages():
            if any(k in e.key for k in TIER_KERNELS):
                us += getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0)
                launches += e.count
        us /= args.calls
        res = {"screened": int(st[0]), "us_per_call": us, "launches_per_call": launches / args.calls}
        if st[0] == 1 and us > 0:
            pairs = (m - min(m, 592 * 128)) * n_pad * nsl
            res["pairs_per_s"] = pairs / (us * 1e-6)
            res["bound_issue_pairs_per_s (assumed)"] = 4 * 148 * SM_CLOCK * 32 / SASS_INSTR_PER_PAIR
            res["bound_mufu_pairs_per_s (assumed)"] = 16 * 148 * SM_CLOCK / 2
        out["cases"][name] = res
        print(name, json.dumps(res), file=sys.stderr)
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
