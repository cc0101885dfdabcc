#!/usr/bin/env python
"""OptimizationMAP on the device (boss_gp_map_multistart, DESIGN.md 2.15) against the mirror's host "lbfgs" driver, on
the same seeded problem and the same starts.

  python tools/bench_map_multistart.py [--reps 3] [--out FILE]

Shapes: n in {128, 512, 2048}, d = 8, y_dim in {1, 4}, M = 32 starts, iters = 40, Matern52, LogNormal priors on all
d + 2 entries of every slice.  Per shape:
  device  OptimizationMAP(algorithm="device") end to end (wall ms, best of --reps), rounds and (slice, start)
          log-likelihood evaluations from BOSS_MS_TRACE, evaluations/s; a torch.profiler run of one solve splits the GPU
          time into the factorisation pipeline and the driver's own kernels (map_prep, map_prior, ms_*);
  host    OptimizationMAP(algorithm="lbfgs") end to end, its rounds (one boss_gp_loglik_grad_batch call per slice and
          round) and evaluations (samples over those calls), evaluations/s;
  batch   boss_gp_loglik_grad_batch alone at the device solve's largest batch (y_dim M samples, host pointers):
          evaluations/s.
Both drivers' best log-likelihoods are reported.  One JSON line, with the card name and power limit it was measured
at."""
import argparse
import json
import os
import re
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

from tools.bench_screen import card  # noqa: E402


class _StderrCapture:
    """fd-level capture of the library's stderr (BOSS_MS_TRACE lines)"""

    def __enter__(self):
        self.f = tempfile.TemporaryFile(mode="w+b")
        sys.stderr.flush()
        self.saved = os.dup(2)
        os.dup2(self.f.fileno(), 2)
        return self

    def __exit__(self, *exc):
        sys.stderr.flush()
        os.dup2(self.saved, 2)
        os.close(self.saved)
        self.f.seek(0)
        self.text = self.f.read().decode(errors="replace")
        self.f.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import boss_b200 as B
    from boss_b200 import _lib
    from tests.util_problems import make_problem
    _lib.init(0)
    d, M, iters = 8, 32, 40
    res = {"card": card(), "d": d, "M": M, "iters": iters, "kernel": "Matern52", "reps": args.reps, "shapes": []}

    def wall(fn):
        best, r = float("inf"), None
        for _ in range(args.reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            r = fn()
            torch.cuda.synchronize()
            best = min(best, (time.perf_counter() - t0) * 1e3)
        return best, r

    for n in (128, 512, 2048):
        for y_dim in (1, 4):
            X, Y, _, _, _ = make_problem(n, d, seed=100 + n + y_dim, y_dim=y_dim)
            model = B.GaussianProcess(kernel=B.Matern52Kernel(),
                                      lengthscale_priors=[B.mvlognormal([0.0] * d, [0.7] * d)] * y_dim,
                                      amplitude_priors=[B.LogNormal(0.0, 0.5)] * y_dim,
                                      noise_std_priors=[B.LogNormal(np.log(0.1), 0.5)] * y_dim)
            dom = B.Domain((np.zeros(d), np.ones(d)))
            prob = B.BossProblem(lambda x: x, dom, B.ExpectedImprovement(B.LinFitness([1.0] + [0.0] * (y_dim - 1))),
                                 model, B.ExperimentData(X, Y))
            sampler = model.params_sampler(np.random.default_rng(7))
            starts = [sampler() for _ in range(M)]

            def run(alg):
                return B.estimate_parameters(B.OptimizationMAP(list(starts), iters=iters, algorithm=alg), prob)

            row = {"n": n, "y_dim": y_dim}
            # device: warm-up, rounds and evaluations from the trace, then the timed runs
            run("device")
            os.environ["BOSS_MS_TRACE"] = "1"
            with _StderrCapture() as cap:
                run("device")
            del os.environ["BOSS_MS_TRACE"]
            m = re.search(r"rounds (\d+) evaluations (\d+)", cap.text)
            rounds, evals = int(m.group(1)), int(m.group(2))
            ms, r = wall(lambda: run("device"))
            row["device"] = {"wall_ms": round(ms, 3), "rounds": rounds, "loglik_evals": evals,
                             "evals_per_s": round(evals / ms * 1e3, 1), "ms_per_round": round(ms / rounds, 3),
                             "best_loglike": r.loglike}
            # GPU time by kernel in one solve (a separate, profiled run)
            from torch.profiler import ProfilerActivity, profile
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                run("device")
                torch.cuda.synchronize()
            own = other = 0.0
            for e in prof.key_averages():
                t = getattr(e, "self_device_time_total", None)
                if t is None:
                    t = getattr(e, "self_cuda_time_total", 0.0)
                if t <= 0:
                    continue
                if e.key.startswith(("void boss::map_", "void boss::ms_", "boss::map_", "boss::ms_")) or \
                        "map_prep_kernel" in e.key or "map_prior_kernel" in e.key or "ms_propose" in e.key or \
                        "ms_advance" in e.key or "ms_init" in e.key:
                    own += t
                else:
                    other += t
            row["device"]["gpu_ms_driver_kernels"] = round(own / 1e3, 3)
            row["device"]["gpu_ms_loglik_pipeline"] = round(other / 1e3, 3)
            # host driver: count its batched calls
            calls = {"n": 0, "S": 0}
            orig = _lib.loglik_grad_batch

            def counted(X_, Ymm, L, *a, **k):
                calls["n"] += 1
                calls["S"] += np.shape(L)[0]
                return orig(X_, Ymm, L, *a, **k)
            _lib.loglik_grad_batch = counted
            try:
                run("lbfgs")
                calls["n"] = calls["S"] = 0
                run("lbfgs")
                hc = dict(calls)
                ms, r = wall(lambda: run("lbfgs"))
            finally:
                _lib.loglik_grad_batch = orig
            row["host"] = {"wall_ms": round(ms, 3), "rounds": hc["n"] // y_dim, "loglik_evals": hc["S"],
                           "evals_per_s": round(hc["S"] / ms * 1e3, 1), "best_loglike": r.loglike}
            # the batch primitive alone at the largest batch of the device solve
            S = y_dim * M
            rng = np.random.default_rng(3)
            L = np.exp(rng.normal(0.0, 0.7, (S, d)))
            A = np.exp(rng.normal(0.0, 0.5, S))
            Nn = np.exp(rng.normal(np.log(0.1), 0.5, S))
            Ys = np.repeat(Y, M, axis=0)
            ms, _ = wall(lambda: _lib.loglik_grad_batch(X, Ys, L, A, Nn, _lib.KERNEL_MATERN52))
            row["loglik_grad_batch"] = {"S": S, "ms": round(ms, 3), "evals_per_s": round(S / ms * 1e3, 1)}
            row["device_speedup"] = round(row["host"]["wall_ms"] / row["device"]["wall_ms"], 2)
            res["shapes"].append(row)
            print(json.dumps(row), file=sys.stderr, flush=True)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
