#!/usr/bin/env python
"""bench.py -- headline benchmark of the BOSS.jl GP hot path on B200 (contract: see DESIGN.md, Measurement).

Workload (BASELINE.json configs[1], per-GPU share): GP posterior + EI scoring + argmax over
M = 2 Mi candidates per GPU, n = 2048 training points, d = 8, Matern52 ARD  (16 Mi candidates at 8 GPUs;
weak scaling, candidates sharded by contiguous block, (best value, index) pairs all-gathered over NCCL).
A "step" = one scoring pass over the rank's candidates.  `value` = candidates/s with candidates resident
in HBM; `e2e` = the same through the host-pointer C-ABI call (pinned host candidates, H2D inside the
timed region, D2H of the argmax pair; `e2e.pageable` = the same from ordinary pageable host memory).  The FP64 roofline
denominator (cuBLAS DGEMM 8192^3) is measured inside this run.  The second headline metric, batched GP log-likelihood evals/s at
n = 2048, d = 8 (S = 256 hyper-parameter vectors per GPU per step), is reported under "loglik".

`--impl reference` times the CPU restatement of the reference path (oracle/, numpy + OpenBLAS with all host
threads) on a bounded sample of the same workload; Julia is not installed, so the reference itself cannot run.

`--dump-outputs DIR` writes, after the timed steps, what each timed path returned to its caller in its last step as
DIR/<name>.npy (float64; argmax indices are stored as float64, exact below 2^53): the (best value, index) pair of the
resident, pinned and pageable EI scoring passes, the S log-likelihoods, and the log-likelihoods and (S, d + 2)
gradients of the value + gradient pass.  Every input is seeded, so two builds run with the same arguments can be
compared output for output.  Under torchrun every rank writes its own files, suffixed _rank<r>.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the benchmark leaves the source tree as it found it (it may be read-only)

N_TRAIN, X_DIM, KERNEL_ID = 2048, 8, 2
M_PER_GPU = 1 << 21
LOGLIK_S_PER_GPU = 256
F_CAND = N_TRAIN * N_TRAIN + N_TRAIN * (3 * X_DIM + 12)                      # SURVEY.md 8(d): 4 268 032 flop / candidate
F_LL = N_TRAIN * (N_TRAIN + 1) // 2 * (3 * X_DIM + 8) + N_TRAIN ** 3 / 3 + N_TRAIN ** 2 + 3 * N_TRAIN  # 2.9347e9
# value + gradient: Cholesky n^3/3, W = L^-1 n^3/3, K^-1 = W^T W n^3/3, kernel + derivative evaluations (6d + 14 each)
F_LLG = N_TRAIN ** 3 + N_TRAIN * (N_TRAIN + 1) // 2 * (6 * X_DIM + 14) + 3 * N_TRAIN ** 2
# the scoring kernel's own share of F_CAND: V = W K* over the triangle (n^2) + the column sums of squares (2n); the
# cross-covariance evaluations (n (3d + 10)) belong to xcov_kernel and count only in the whole-step fraction
F_TRMM = N_TRAIN * N_TRAIN + 2 * N_TRAIN                                     # 4 198 400 flop / candidate
CPU_SAMPLE_M = 8192


def fp64_peak_static():
    """cuBLAS DGEMM TFLOP/s measured on this pool's B200 in round 1 (profiles/fp64_peaks_r01.json); MEASURED_PEAKS.json
    only carries HBM and bf16 figures.  Used only if the in-run measurement below fails."""
    try:
        with open(os.path.join(ROOT, "profiles", "fp64_peaks_r01.json")) as f:
            return float(json.load(f)["fp64_tflops_peak_used"]), "round-1 file profiles/fp64_peaks_r01.json (cuBLAS DGEMM 8192^3)"
    except Exception:
        return 37.0, "fallback: nominal B200 FP64 (no measured DGEMM file)"


def measure_dgemm_peak(torch, sustained_s=3.0):
    """The FP64 roofline denominator, measured in THIS run: cuBLAS DGEMM 8192^3 through torch.matmul(float64), CUDA events
    on torch's current stream.  burst = best of 10 single GEMMs; sustained = back-to-back GEMMs for `sustained_s` seconds."""
    n = 8192
    a = torch.rand((n, n), dtype=torch.float64, device="cuda"); b = torch.rand((n, n), dtype=torch.float64, device="cuda")
    c = torch.empty((n, n), dtype=torch.float64, device="cuda")
    flop = 2.0 * n ** 3
    for _ in range(3):
        torch.matmul(a, b, out=c)
    torch.cuda.synchronize()
    best = 0.0
    for _ in range(10):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); torch.matmul(a, b, out=c); e1.record(); torch.cuda.synchronize()
        best = max(best, flop / (e0.elapsed_time(e1) * 1e-3) * 1e-12)
    per = flop / (best * 1e12)
    reps = max(4, int(sustained_s / per))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        torch.matmul(a, b, out=c)
    e1.record(); torch.cuda.synchronize()
    sus = flop * reps / (e0.elapsed_time(e1) * 1e-3) * 1e-12
    del a, b, c
    torch.cuda.empty_cache()
    return {"burst_tflops": best, "sustained_tflops": sus, "sustained_reps": reps,
            "how": "cuBLAS DGEMM 8192^3 via torch.matmul(float64), CUDA events, in this run"}


def make_problem():
    from tests.util_problems import make_problem as mp
    X, Y, ls, amp, ns = mp(N_TRAIN, X_DIM, seed=1002)
    return X, Y[0], ls[0], float(amp[0]), float(ns[0])


# ---------------------------------------------------------------------------------------------
# reference arm / CPU baseline (oracle port on host cores)
# ---------------------------------------------------------------------------------------------
def cpu_threads():
    try:
        from threadpoolctl import threadpool_info
        return max([p.get("num_threads", 1) for p in threadpool_info()] + [1])
    except Exception:
        return os.cpu_count() or 1


def use_all_host_threads():
    """torchrun exports OMP_NUM_THREADS=1 for every rank; the CPU arm is meant to use every host core."""
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=os.cpu_count() or 1)
    except Exception:
        pass


def cpu_score_once(post, Xs, best):
    """-> (best value, index), the pair the GPU path returns."""
    from oracle import boss_oracle as O
    acq, _, _ = O.ei_acquisition([[post]], Xs, [1.0], best, None)
    bi = O.julia_argmax_fast(acq)
    return float(acq[bi]), bi


def dump_outputs(out_dir, outputs, suffix=""):
    """Each output as out_dir/<name><suffix>.npy in float64."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in outputs.items():
        np.save(os.path.join(out_dir, name + suffix + ".npy"), np.asarray(a, dtype=np.float64))


def cpu_baseline(budget_s=12.0):
    """Mode B (best-case CPU: the reference's matrix API mean_and_var(post, X::Matrix),
    src/models/gaussian_process.jl:174-178, level-3 BLAS on all host threads) on CPU_SAMPLE_M-candidate tiles,
    plus mode A (the access pattern BOSS.jl ships: one candidate per call, expected_improvement.jl:74-84)."""
    from oracle import boss_oracle as O
    use_all_host_threads()
    X, y, ls, amp, ns = make_problem()
    post = O.posterior_fit(X, y, ls, amp, ns, KERNEL_ID)
    best = float(np.max(y))
    rng = np.random.default_rng(2002)
    Xs = rng.random((X_DIM, CPU_SAMPLE_M))
    cpu_score_once(post, Xs[:, :512], best)
    t0 = time.perf_counter(); reps = 0
    while True:
        cpu_score_once(post, Xs, best); reps += 1
        if time.perf_counter() - t0 > budget_s * 0.6 or reps >= 8:
            break
    tB = (time.perf_counter() - t0) / reps
    t0 = time.perf_counter(); k = 0
    while time.perf_counter() - t0 < budget_s * 0.2 and k < 2000:
        cpu_score_once(post, Xs[:, k % CPU_SAMPLE_M][:, None], best); k += 1
    tA = (time.perf_counter() - t0) / max(k, 1)
    L, A, N = np.full((1, X_DIM), 0.7), np.array([1.0]), np.array([0.1])
    t0 = time.perf_counter(); r = 0
    while time.perf_counter() - t0 < budget_s * 0.2 and r < 20:
        O.gp_loglik_batch(X, y, L, A, N, KERNEL_ID); r += 1
    tL = (time.perf_counter() - t0) / max(r, 1)
    return {"value": CPU_SAMPLE_M / tB, "unit": "candidates/s", "cores": cpu_threads(), "kind": "port",
            "sample": f"{reps} x {CPU_SAMPLE_M}-candidate batched tiles (level-3 BLAS, mode B) of the n=2048,d=8 Matern52 "
                      f"EI scoring workload; restated reference path (numpy/OpenBLAS) - Julia is not installed",
            "one_candidate_per_call_value": 1.0 / tA, "loglik_evals_per_s": 1.0 / tL,
            "host_cpus": os.cpu_count()}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import boss_oracle as O
    use_all_host_threads()
    X, y, ls, amp, ns = make_problem()
    post = O.posterior_fit(X, y, ls, amp, ns, KERNEL_ID)
    best = float(np.max(y))
    Xs = np.random.default_rng(2002).random((X_DIM, CPU_SAMPLE_M))
    for _ in range(args.warmup):
        cpu_score_once(post, Xs[:, :2048], best)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        res = cpu_score_once(post, Xs, best)
    dt = (time.perf_counter() - t0) / args.steps
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"ei_best_value": [res[0]], "ei_best_index": [res[1]]})
    val = CPU_SAMPLE_M / dt
    # mode A beside it: what BOSS.jl's maximizers actually do - one candidate per call (grid.jl:52-53)
    t1 = time.perf_counter(); k = 0
    while time.perf_counter() - t1 < 3.0 and k < 2000:
        cpu_score_once(post, Xs[:, k % CPU_SAMPLE_M][:, None], best); k += 1
    mode_a = k / (time.perf_counter() - t1)
    cb = {"value": val, "unit": "candidates/s", "cores": cpu_threads(), "kind": "port",
          "sample": f"each step = one {CPU_SAMPLE_M}-candidate batched tile (mode B, level-3 BLAS, all host threads) of the "
                    f"2 Mi-candidate per-GPU workload; oracle port - the Julia reference cannot run in this image",
          "one_candidate_per_call_value": mode_a,
          "note": "mode B (batched matrix API) is the best case for the CPU; mode A is the access pattern BOSS.jl ships"}
    print(file=args.out, flush=True, *[json.dumps({
        "impl": "reference", "metric": "EI candidate evals/sec (n=2048,d=8)", "value": val, "unit": "candidates/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": dict(workload_config(args.gpus), candidates_per_step=CPU_SAMPLE_M,
                       reference_sample="one 8192-candidate tile per step (a bounded sample of the 2 Mi-candidate share; "
                                        "throughput is per candidate, so the sample size does not change it)"),
        "cpu_baseline": cb,
        "e2e": {"value": val, "unit": "candidates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})])


def workload_config(n_gpus):
    return {"workload": "BASELINE configs[1] per-GPU share: GP posterior + EI grid scoring + argmax, n=2048 train pts, "
                        "d=8, Matern52 ARD, 2 Mi candidates per GPU (16 Mi at 8 GPUs)",
            "n_train": N_TRAIN, "x_dim": X_DIM, "kernel": "Matern52", "candidates_per_gpu": M_PER_GPU,
            "candidates_total": M_PER_GPU * n_gpus, "sharding": f"candidate-block x{n_gpus}",
            "l2_policy": "inputs larger than L2 (128 MiB candidates + 1.2 GB K* scratch streamed per step; 126 MB L2)"}


# ---------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                       "-i", str(gpu_index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush(); self.f.seek(0)
        sm, mx, reasons = [], [], set()
        for line in self.f.read().splitlines():
            c = [t.strip() for t in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1])); mx.append(float(c[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if sm:
            out = {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        return out


# ---------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------
def run_gpu(args):
    import torch
    import torch.distributed as dist
    import boss_b200  # noqa: F401
    from boss_b200 import _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    _lib.init(local)
    lib_stream = torch.cuda.ExternalStream(_lib.stream_ptr(), device=torch.device("cuda", local))

    X, y, ls, amp, ns = make_problem()
    gp = _lib.gp_fit(X, y, ls, amp, ns, KERNEL_ID)          # deterministic: bit-identical replica on every rank
    assert gp is not None
    fit_ms = []
    for _ in range(5):                                       # posterior fit latency (amortised over the scoring passes)
        t0 = time.perf_counter(); g2 = _lib.gp_fit(X, y, ls, amp, ns, KERNEL_ID); fit_ms.append((time.perf_counter() - t0) * 1e3)
        g2.free()
    best = float(np.max(y))
    M = M_PER_GPU
    gen = torch.Generator(device="cuda"); gen.manual_seed(2002 + rank)
    Xs_dev = torch.rand((M, X_DIM), dtype=torch.float64, device="cuda", generator=gen)   # = d x M column-major
    Xs_host = torch.empty((M, X_DIM), dtype=torch.float64, pin_memory=True)
    Xs_host.copy_(Xs_dev)
    Xs_np = Xs_host.numpy().T                                 # d x M view, no copy (pinned)
    Xs_pageable = np.array(Xs_host.numpy(), copy=True).T      # ordinary pageable memory: what a Julia Matrix{Float64} is

    # loglik workload: S hyper-parameter vectors per GPU
    from tests.util_problems import make_hyper_samples
    S = LOGLIK_S_PER_GPU
    Lh, Ah, Nh = make_hyper_samples(S, X_DIM, seed=3003 + rank)
    t_X = torch.tensor(np.ascontiguousarray(X.T), device="cuda"); t_y = torch.tensor(y, device="cuda")
    t_L = torch.tensor(Lh, device="cuda"); t_A = torch.tensor(Ah, device="cuda"); t_N = torch.tensor(Nh, device="cuda")
    t_ll = torch.empty(S, dtype=torch.float64, device="cuda")
    t_gr = torch.empty((S, X_DIM + 2), dtype=torch.float64, device="cuda")

    gathered = [torch.zeros(2, dtype=torch.float64, device="cuda") for _ in range(world)]
    last_pairs = []          # (best value, global index) of every rank in the last reduction

    def reduce_pairs(bv, bi):
        """(best value, global index) all-gather + deterministic local reduce (NCCL has no arg-max op)."""
        if world == 1:
            return bv, bi
        mine = torch.tensor([bv, float(rank * M + bi)], dtype=torch.float64, device="cuda")
        dist.all_gather(gathered, mine)
        vals = torch.stack(gathered).cpu().numpy()
        last_pairs[:] = vals.tolist()
        k = 0
        for r in range(1, world):
            a, b = vals[k, 0], vals[r, 0]
            if (np.isnan(b) and not np.isnan(a)) or b > a:
                k = r
        return float(vals[k, 0]), int(vals[k, 1])

    def step_resident():
        bv, bi = _lib.ei_score_dev([gp], 1, 1, Xs_dev.data_ptr(), M, [1.0], best, None)
        return reduce_pairs(bv, bi)

    def step_e2e():
        acq, bv, bi = _lib.ei_score([gp], 1, 1, Xs_np, [1.0], best, None, want_acq=False)
        return reduce_pairs(bv, bi)

    def step_e2e_pageable():
        acq, bv, bi = _lib.ei_score([gp], 1, 1, Xs_pageable, [1.0], best, None, want_acq=False)
        return reduce_pairs(bv, bi)

    def step_loglik():
        _lib.loglik_batch_dev(t_X.data_ptr(), X_DIM, N_TRAIN, t_y.data_ptr(), 0, t_L.data_ptr(), t_A.data_ptr(),
                              t_N.data_ptr(), KERNEL_ID, S, t_ll.data_ptr())

    def step_loglik_grad():
        _lib.loglik_grad_batch_dev(t_X.data_ptr(), X_DIM, N_TRAIN, t_y.data_ptr(), 0, t_L.data_ptr(), t_A.data_ptr(),
                                   t_N.data_ptr(), KERNEL_ID, S, t_ll.data_ptr(), t_gr.data_ptr())

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = _lib.launch_count()
        e0.record(lib_stream)
        for _ in range(steps):
            out = fn()
        e1.record(lib_stream)
        barrier()
        ms = e0.elapsed_time(e1)
        launches = _lib.launch_count() - l0
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms / steps, launches, out

    suffix = f"_rank{rank}" if world > 1 else ""
    if args.only == "loglik":          # profiling aid: only the batched log-likelihood step
        ms_ll, launches_ll, _ = timed(step_loglik, args.steps, args.warmup)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"loglik": t_ll.cpu().numpy()}, suffix)
        if rank == 0:
            print(json.dumps({"only": "loglik", "ms_per_step": ms_ll, "evals_per_s": S * world / (ms_ll * 1e-3),
                              "gpu_launches": int(launches_ll)}), file=args.out, flush=True)
        return
    sampler = ClockSampler(local) if rank == 0 else None
    _lib.set_timing(True)
    ms_step, launches, res = timed(step_resident, args.steps, args.warmup)
    trmm_ms, trmm_cnt = _lib.last_kernel_ms(0)               # score_trmm launches of the LAST step
    xcov_ms, xcov_cnt = _lib.last_kernel_ms(1)
    _lib.set_timing(False)
    ms_e2e, _, res_e2e = timed(step_e2e, args.steps, args.warmup)
    ms_e2e_pg, _, res_e2e_pg = timed(step_e2e_pageable, max(2, args.steps // 2), 3)
    ms_ll, launches_ll, _ = timed(step_loglik, max(2, args.steps // 2), 3)   # 4 concurrent sub-batch streams
    _lib.set_timing(True)                                                     # per-kernel-class events: one stream
    ms_ll_serial, _, _ = timed(step_loglik, 2, 3)
    chol_ms, chol_cnt = _lib.last_kernel_ms(2)
    _lib.set_timing(False)
    ll_out = t_ll.cpu().numpy()                                               # step_loglik_grad overwrites t_ll
    ms_llg, launches_llg, _ = timed(step_loglik_grad, max(2, args.steps // 2), 3)
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {
            "ei_best_value": [res[0]], "ei_best_index": [res[1]],
            "ei_e2e_best_value": [res_e2e[0]], "ei_e2e_best_index": [res_e2e[1]],
            "ei_e2e_pageable_best_value": [res_e2e_pg[0]], "ei_e2e_pageable_best_index": [res_e2e_pg[1]],
            "loglik": ll_out, "loglik_grad_value": t_ll.cpu().numpy(), "loglik_grad": t_gr.cpu().numpy()}, suffix)
    # one candidate per call -- the access pattern of the reference's stock maximizers (acq(x) inside NLopt / Optim,
    # grid.jl:52-53): host-pointer C-ABI calls, wall time per call (H2D of the point, all kernels, D2H of the result)
    x1 = np.ascontiguousarray(Xs_pageable[:, :1])
    single = {}
    for name, fn in (("value", lambda: _lib.ei_score([gp], 1, 1, x1, [1.0], best, None)),
                     ("value_grad", lambda: _lib.ei_value_grad([gp], 1, 1, x1, [1.0], best, None))):
        for _ in range(20):
            fn()
        t0 = time.perf_counter()
        for _ in range(200):
            fn()
        single[name + "_call_us"] = (time.perf_counter() - t0) / 200 * 1e6
    single["value_calls_per_s"] = 1e6 / single["value_call_us"]
    try:
        dg = measure_dgemm_peak(torch)          # every rank (keeps the ranks in step); rank 0 reports
    except Exception as e:                      # noqa: BLE001
        dg = {"error": repr(e)}
    cfgs = None
    if not args.no_configs:
        # per-GPU shares of BASELINE configs C3 / C4 / C5 (device-resident, oracle parity spot checks inside); at N > 1
        # every rank runs its share and the times are the max over ranks
        from tools import bench_configs
        cfgs = bench_configs.run_all(torch, _lib, lib_stream, steps=3, dist=dist if world > 1 else None, world=world,
                                     peak_tflops=dg.get("burst_tflops"))

    if rank == 0:
        if "burst_tflops" in dg:
            peak, peak_src = dg["burst_tflops"], ("cuBLAS DGEMM 8192^3 measured in this run (burst = best of 10; the "
                                                  "sustained figure is in roofline.dgemm)")
        else:
            peak, peak_src = fp64_peak_static()
        per_launch_cands = M / max(trmm_cnt, 1)
        achieved = F_TRMM * per_launch_cands / (trmm_ms / max(trmm_cnt, 1) * 1e-3) * 1e-12
        ll_val = S * world / (ms_ll * 1e-3)
        out = {
            "metric": "EI candidate evals/sec (n=2048,d=8)", "value": M * world / (ms_step * 1e-3), "unit": "candidates/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(world),
            "e2e": {"value": M * world / (ms_e2e * 1e-3), "unit": "candidates/s",
                    "h2d_bytes_per_step": M * X_DIM * 8, "d2h_bytes_per_step": 24, "ms_per_step": ms_e2e,
                    "host_memory": "pinned",
                    "pageable": {"value": M * world / (ms_e2e_pg * 1e-3), "ms_per_step": ms_e2e_pg,
                                 "what": "the same call with the candidates in ordinary pageable memory (a Julia "
                                         "Matrix{Float64}): the library stages them through two pinned slots on a copy "
                                         "stream while the previous chunk computes",
                                 "argmax_index": res_e2e_pg[1]}},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {"bound": "tensor", "kernel": "score_trmm_kernel (FP64 DMMA.8x8x4)", "achieved": achieved,
                         "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak, "traffic": None,
                         "peak_source": peak_src, "launches_timed": trmm_cnt, "avg_launch_ms": trmm_ms / max(trmm_cnt, 1),
                         "flop_per_candidate": F_TRMM, "step_flop_per_candidate": F_CAND,
                         "candidates_per_launch": per_launch_cands,
                         "xcov_ms_per_step": xcov_ms, "trmm_ms_per_step": trmm_ms,
                         "whole_step_frac": F_CAND * M / (ms_step * 1e-3) * 1e-12 / peak,
                         "dgemm": dg, "dgemm_round1_file": fp64_peak_static()[0],
                         # the second headline metric and the per-config numbers, repeated here because only the contract's
                         # keys of this line are carried into the driver's summary
                         "loglik": {"evals_per_s": ll_val, "ms_per_step": ms_ll,
                                    "frac_of_peak": F_LL * S / (ms_ll * 1e-3) * 1e-12 / peak},
                         "loglik_grad": {"evals_per_s": S * world / (ms_llg * 1e-3),
                                         "frac_of_peak": F_LLG * S / (ms_llg * 1e-3) * 1e-12 / peak},
                         "configs": [{k: c[k] for k in c if k in ("config", "kernel", "frac_of_dgemm_peak",
                                                                  "frac_of_dgemm_peak_value_grad", "ms_per_step",
                                                                  "loglik_evals_per_s", "candidates_per_s",
                                                                  "on_device_multistart_frac", "n_gpus")}
                                     for c in (cfgs or [])]},
            "loglik": {"metric": "GP loglik evals/sec (n=2048,d=8)", "value": ll_val, "unit": "evals/s",
                       "samples_per_gpu_per_step": S, "ms_per_step": ms_ll, "flop_per_eval": F_LL,
                       "achieved_tflops_per_gpu": F_LL * S / (ms_ll * 1e-3) * 1e-12,
                       "frac_of_peak": F_LL * S / (ms_ll * 1e-3) * 1e-12 / peak,
                       "single_stream_ms_per_step": ms_ll_serial, "chol_gemm_ms_per_step_single_stream": chol_ms,
                       "chol_gemm_launches": chol_cnt, "gpu_launches": int(launches_ll)},
            "loglik_grad": {"metric": "GP loglik + hyper-parameter gradient evals/sec (n=2048,d=8)",
                            "value": S * world / (ms_llg * 1e-3), "unit": "evals/s", "ms_per_step": ms_llg,
                            "flop_per_eval": F_LLG, "achieved_tflops_per_gpu": F_LLG * S / (ms_llg * 1e-3) * 1e-12,
                            "frac_of_peak": F_LLG * S / (ms_llg * 1e-3) * 1e-12 / peak, "gpu_launches": int(launches_llg)},
            "single_point": dict(single, what="one candidate per host call through boss_ei_score / boss_ei_value_grad "
                                              "(n=2048, d=8); cpu_baseline.one_candidate_per_call_value is the CPU port's rate"),
            "fit": {"what": "boss_gp_fit wall time (host call: H2D of X, y; K, Cholesky, W = L^-1, alpha; n=2048, d=8)",
                    "ms_median": float(np.median(fit_ms)), "flop": F_LL + N_TRAIN ** 3 / 3},
            "argmax": {"value": res[0], "index": res[1], "e2e_index": res_e2e[1], "per_rank_pairs": list(last_pairs)},
        }
        try:
            with open(os.path.join(ROOT, "profiles", "score_trmm_traffic.json")) as f:
                out["roofline"]["traffic"] = json.load(f)["dram_bytes_per_launch"]
        except Exception:
            pass
        if cfgs is not None:
            out["configs"] = cfgs
        if world == 1 and not args.no_cpu_baseline:
            out["cpu_baseline"] = cpu_baseline()
        print(json.dumps(out), file=args.out, flush=True)
    gp.free()
    if world > 1:
        dist.destroy_process_group()


class StdoutToStderr:
    """The contract is ONE JSON line on stdout.  NCCL (`NCCL version ...` with NCCL_DEBUG set) and other native
    libraries write to file descriptor 1 directly; route fd 1 to stderr while the benchmark runs and hand the
    real stdout back only to the final print."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)
        self.real = os.fdopen(self.saved, "w")
        return self.real

    def __exit__(self, *exc):
        sys.stdout.flush()
        self.real.flush()
        os.dup2(self.real.fileno(), 1)
        return False


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the C3/C4/C5 per-config numbers (N=1 only)")
    ap.add_argument("--only", default="all", choices=["all", "loglik"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs to DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    with StdoutToStderr() as real_stdout:
        args.out = real_stdout
        if args.impl == "reference":
            run_reference(args)
        else:
            run_gpu(args)


if __name__ == "__main__":
    main()
