#!/usr/bin/env python
"""The mean tiers of argmax screening (DESIGN.md 2.9), alternated in one process.

  python tools/bench_screen_tiers.py [--rounds 3] [--steps 3] [--out FILE] [--profile FILE]

Tiers: "f64" (BOSS_SCREEN_F64=1 BOSS_SCREEN_NO_RESEED=1, the FP64 means of every candidate), "f32" (the FP32 tier,
BOSS_SCREEN_NO_RESEED=1) and "f32_reseed" (the default).  Cases: bench.py's problem (n = 2048, d = 8, Matern52, 2 Mi
candidates) with the candidates resident on the device, in pinned and in pageable host memory; C5's shape (n = 1024,
d = 10, 4 outputs, EI x PoF, 512 Ki candidates, argmax only); and the bench problem refitted with noise 1e-4, where
the larger sum |alpha| widens E and more candidates need the FP64 refinement.  Each round times `steps` calls of every
tier in turn; printed per case and tier: ms per call, kernel launches per call, pool size, ambiguous candidates, and
whether the (value, index) pairs are bit-identical to the f64 tier's.  One JSON line, with the card name and power limit
it was measured at.
--profile FILE: afterwards, one resident bench call per tier under torch.profiler (a run of its own, after the timed
rounds); the CUDA time per kernel name and tier goes to FILE as JSON, with the FP32 tier's mean kernel per chunk and
its (candidate, training point) pairs per second beside two bounds whose rates are assumptions, not measurements, the
call's kernel timeline with streams, the kernels that start inside the FP32 pass's span, and the variance tier's rows
in and out."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CH0 = 75_776                 # the first chunk of the bench problem (FP64 tier), candidates
SASS_INSTR_PER_PAIR = 10.6   # the MMA mean loop at DP = 8: 676 instructions per 64 pairs a thread (cuobjdump -sass)
MUFU_PER_PAIR = 2            # rsqrt and ex2 (Matern52)
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
    ap.add_argument("--profile", default=None)
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
    gp_ill = _lib.gp_fit(X, Y[0], ls[0], amp[0], 1e-4, _lib.KERNEL_MATERN52)

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
        "bench_noise_1e-4": (M, lambda: _lib.ei_score_dev([gp_ill], 1, 1, Xs_dev.data_ptr(), M, [1.0], best, None)),
    }

    def timed(fn, steps):
        fn()                                     # warm-up (and this mode's scratch sizes)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(steps):
            r = fn()
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) / steps * 1e3, r

    tiers = {"f64": ("BOSS_SCREEN_F64", "BOSS_SCREEN_NO_RESEED"), "f32": ("BOSS_SCREEN_NO_RESEED",), "f32_reseed": ()}
    out = {"card": card(), "rounds": args.rounds, "steps": args.steps, "cases": {}}
    for name, (m, fn) in cases.items():
        ms = {t: [] for t in tiers}
        info, same = {}, True
        for _ in range(args.rounds):
            ref = None
            for t, env in tiers.items():
                for k in ("BOSS_SCREEN_F64", "BOSS_SCREEN_NO_RESEED"):
                    os.environ.pop(k, None)
                for k in env:
                    os.environ[k] = "1"
                ms_t, r = timed(fn, args.steps)
                ms[t].append(ms_t)
                st, amb, var = _lib.dbg_screen_stats(), _lib.dbg_screen_ambiguous(), _lib.dbg_screen_var()
                l0 = _lib.launch_count()
                fn()
                info[t] = {"screen_state": st[0], "bounded": st[1], "pool": st[2], "ambiguous": amb[0],
                           "var_tier_rows_in_out": list(var), "launches_per_call": _lib.launch_count() - l0}
                key = (np.float64(r[0]).view(np.int64), r[1])
                ref = key if ref is None else ref
                same = same and key == ref
        for k in ("BOSS_SCREEN_F64", "BOSS_SCREEN_NO_RESEED"):
            os.environ.pop(k, None)
        out["cases"][name] = {
            "M": m, "ms": ms, "ms_median": {t: float(np.median(v)) for t, v in ms.items()},
            "ms_spread": {t: float(np.max(v) - np.min(v)) for t, v in ms.items()},
            "speedup_vs_f64_median": {t: float(np.median(ms["f64"]) / np.median(v)) for t, v in ms.items()},
            "tiers": info, "pairs_bit_identical": bool(same)}
        print(name, json.dumps(out["cases"][name]), file=sys.stderr, flush=True)
    if args.profile:
        from torch.profiler import ProfilerActivity, profile
        prof_out = {"card": out["card"], "case": "bench_resident", "tiers": {}}
        fn = cases["bench_resident"][1]
        for t, env in tiers.items():
            for k in ("BOSS_SCREEN_F64", "BOSS_SCREEN_NO_RESEED"):
                os.environ.pop(k, None)
            for k in env:
                os.environ[k] = "1"
            fn()
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as pr:
                fn()
                torch.cuda.synchronize()
            ker = {}
            # the call's kernels in start order (device clock, us from the first), with the stream they ran on: the
            # device-resident FP32 pass runs on a side stream beside the first chunk's kernels
            evs = sorted((e for e in pr.events() if e.device_type.name == "CUDA"), key=lambda e: e.time_range.start)
            t0 = evs[0].time_range.start if evs else 0
            tl = [{"name": e.name[:80], "start_us": e.time_range.start - t0, "dur_us": e.time_range.end - e.time_range.start,
                   "stream": getattr(e, "device_resource_id", None)} for e in evs]
            prof_out.setdefault("timeline", {})[t] = tl
            span = [(x["start_us"], x["start_us"] + x["dur_us"]) for x in tl if "screen_mean_bound_kernel" in x["name"]]
            if span:
                a0, a1 = span[0]
                inside = [x for x in tl if "screen_mean_bound_kernel" not in x["name"] and a0 <= x["start_us"] < a1]
                prof_out.setdefault("inside_fp32_pass", {})[t] = {
                    "pass_us": [a0, a1], "kernels_started_inside": len(inside),
                    "kernel_us_inside": sum(min(x["dur_us"], a1 - x["start_us"]) for x in inside),
                    "names": sorted({x["name"] for x in inside})}
            prof_out.setdefault("var_tier_rows_in_out", {})[t] = list(_lib.dbg_screen_var())
            for e in pr.key_averages():
                if e.device_type.name == "CUDA" or getattr(e, "cuda_time_total", 0) > 0:
                    us = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0)
                    if us > 0:
                        ker[e.key] = {"us": us, "count": e.count}
            prof_out["tiers"][t] = dict(sorted(ker.items(), key=lambda kv: -kv[1]["us"])[:25])
            mean_k = [(k, v) for k, v in ker.items() if "screen_mean_bound_kernel" in k]
            if mean_k:
                k, v = mean_k[0]
                per_chunk = v["us"] / v["count"]   # one launch over every candidate after the first chunk
                pairs = (M - CH0) * 2048                 # every candidate after the first chunk, n = 2048
                clk = 1.965e9                            # the card's maximum SM clock (sm_max_clock)
                prof_out["tiers"][t]["mean_tier"] = {
                    "kernel": k, "us_per_chunk": per_chunk, "chunks": v["count"],
                    "pairs_per_s": pairs / (v["us"] * 1e-6),
                    "bound_issue_pairs_per_s (assumed: 1 warp instruction / clock / SM sub-partition, "
                    "SASS_INSTR_PER_PAIR from cuobjdump)": 4 * 148 * clk * 32 / SASS_INSTR_PER_PAIR,
                    f"bound_mufu_pairs_per_s (assumed: 16 MUFU results / clock / SM, {MUFU_PER_PAIR} per pair)":
                        16 * 148 * clk / MUFU_PER_PAIR}
        for k in ("BOSS_SCREEN_F64", "BOSS_SCREEN_NO_RESEED"):
            os.environ.pop(k, None)
        with open(args.profile, "w") as f:
            json.dump(prof_out, f)
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
