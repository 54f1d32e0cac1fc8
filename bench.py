#!/usr/bin/env python
"""bench.py -- dog-leg iterations/sec of libdogleg-b200 on N B200s, with roofline and CPU baseline.

Headline: the mrcal-shaped sparse config (C2 of SURVEY.md section 8; BASELINE.json configs[1]).
One "step" = one complete solve of the synthetic problem through the public API
(dogleg_gpu_optimize_sparse for `value`: device-resident inputs; dogleg_optimize2 with HOST
callbacks and pinned H2D for `e2e`); the metric is accepted dog-leg iterations per second of
library time. The user callback body (the synthetic model) is excluded from `e2e` on both arms
(it is user code and identical for both); for `value` the callback is a kernel on the solver's
stream and is included (`value_excl_callback` subtracts its measured time).

Without --config the line also carries `extra_configs`: short runs of c3 (batched dense), c4 (bundle
adjustment; single GPU only unless --extras all) and c5 (large dense), each with its own
value / e2e / roofline / clocks, at the same number of GPUs -- and a `parity` block: the reference
solved to convergence once on the same problem, compared with what the GPU arm returned.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                  [--config c2|c2s|c3|c4|c4m|c4s|c5] [--extras default|all|none] [--dump-outputs DIR]

  c2   mrcal-shaped calibration, Nstate 1268, Nmeas 1e6 (default)      c3  100 000 batched dense 256x16
  c4   bundle adjustment, 10 k cameras x 1 M points (c4m / c4s: 1/10, 1/100 scale)
  c5   dense 500 000 x 4096

N>1 (torchrun): one process per GPU.
  c2 (headline): `value` / `e2e` = N independent solves of the problem at the same time, one per GPU, no
      communication ("scaling": "weak"): a C2-sized iteration is 0.4 ms of which half is a dependency chain
      that does not shard (DESIGN.md section 7). The row-sharded solve of ONE problem over the N GPUs
      (dogleg_gpu_optimize_sparse_sharded: each rank evaluates its frames -- over its own PCIe link in the
      e2e leg -- and one grouped ncclAllReduce per evaluation sums the partials) is measured in the same run
      and reported as `sharded` (strong scaling) with its collective count and bytes.
  c4 / c5: ONE problem, measurements row-sharded (dogleg_gpu_optimize_sparse_sharded /
      dogleg_gpu_optimize_dense_sharded); strong scaling.
  c3: the batch of independent problems is split over the GPUs, no communication.
torch.distributed only carries the NCCL unique id, the
barrier and the max-over-ranks of the timings.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

CONFIGS = {
    # name: (ncam, nframes, npts)  -> Nstate = 12c + 6(c-1) + 6f + 2, Nmeas = 2 c f k
    "c2":  (4, 200, 625),      # Nstate 1268, Nmeas 1,000,000, nnz 22.5M  (BASELINE.json configs[1])
    "c2s": (4, 40, 125),       # small variant for quick checks
    # bundle adjustment (BASELINE.json configs[3]): ("ba", cameras, points, observations/point, window, long-range permille)
    "c4":  ("ba", 10000, 1000000, 4, 32, 0),   # Nstate 3,090,000, Nmeas 8,000,000, nnz 96M
    "c4m": ("ba", 1000, 100000, 4, 32, 0),     # 1/10 scale
    "c4s": ("ba", 100, 10000, 4, 32, 0),       # 1/100 scale
}


def make_problem(H, cfg):
    c = CONFIGS[cfg]
    if c[0] == "ba":
        return H.Problem.ba(c[1], c[2], c[3], c[4], c[5], seed=4)
    return H.Problem.mrcal(c[0], c[1], c[2], seed=2)


def shard_alignment(cfg):
    """columns that must stay on one rank: a whole frame (mrcal) / all observations of a point (ba)"""
    c = CONFIGS[cfg]
    return 2 * c[3] if c[0] == "ba" else 2 * c[0] * c[2]


def measured_traffic(cfg, kernel):
    """DRAM bytes per launch of the named kernel from the committed ncu captures (profiles/traffic_r01.json)."""
    for name in ("traffic_r02.json", "traffic_r01.json"):
        try:
            v = json.load(open(os.path.join(ROOT, "profiles", name))).get(cfg, {}).get(kernel)
        except (OSError, ValueError):
            v = None
        if v is not None:
            return v
    return None


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return float(d["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons DURING the timed region (B200_PROFILING.md), sampled through
    NVML every 20 ms (the same counters `nvidia-smi --query-gpu=clocks.sm,clocks_event_reasons.*` prints)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.sm, self.reasons, self.stop_flag, self.max_sm = index, [], set(), False, None
        self.ready = threading.Event()

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(visible.split(",")[self.index]) if visible and visible.split(",")[self.index].isdigit() else self.index
            h = nv.nvmlDeviceGetHandleByIndex(idx)
            self.max_sm = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            names = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                     "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                     "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                     "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)}
            get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
                getattr(nv, "nvmlDeviceGetCurrentClocksThrottleReasons")
            while not self.stop_flag:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                mask = int(get_reasons(h))
                for n, bit in names.items():
                    if mask & bit:
                        self.reasons.add(n)
                self.ready.set()
                time.sleep(0.02)
        except Exception as ex:          # pragma: no cover - keep the bench alive without NVML
            self.error = str(ex)
            self.ready.set()

    def wait_first(self, timeout=5.0):
        self.ready.wait(timeout)

    def finish(self):
        self.stop_flag = True
        self.join(timeout=2.0)
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.max_sm,
                "reasons": sorted(self.reasons), "samples": len(self.sm)}


def dist_setup(ngpus):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl" if torch.cuda.is_available() else "gloo")
    return rank, world, local, dist


def barrier_max(dist, seconds):
    """max over ranks of a timing (the contract: time = max over ranks)."""
    if dist is None:
        return seconds
    import torch
    dev = "cuda" if torch.cuda.is_available() else "cpu"
    t = torch.tensor([seconds], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def barrier_sum(dist, v):
    if dist is None:
        return v
    import torch
    dev = "cuda" if torch.cuda.is_available() else "cpu"
    t = torch.tensor([v], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return float(t.item())


def nccl_setup(L, rank, world, dist):
    """NCCL communicator of the library itself; torch.distributed only ships the unique id."""
    import torch
    L.dogleg_gpu_nccl_get_unique_id.argtypes = [C.c_void_p]
    L.dogleg_gpu_nccl_init.argtypes = [C.c_int, C.c_int, C.c_void_p]
    uid = torch.zeros(128, dtype=torch.uint8)
    if rank == 0:
        buf = (C.c_ubyte * 128)()
        assert L.dogleg_gpu_nccl_get_unique_id(buf) == 0, L.dogleg_gpu_last_error()
        uid = torch.tensor(list(buf), dtype=torch.uint8)
    uid = uid.cuda()
    dist.broadcast(uid, 0)
    idb = (C.c_ubyte * 128)(*uid.cpu().tolist())
    assert L.dogleg_gpu_nccl_init(rank, world, idb) == 0, L.dogleg_gpu_last_error()


def cpu_batched_sample(H, N, M, nsample, nthreads):
    """nsample problems of the C3 batch through the reference's dense path on nthreads host threads;
    returns (accepted-or-evaluated iterations, seconds)."""
    import concurrent.futures as cf
    use_ref = H.reference_lib() is not None

    def work(lo, hi):
        acc = 0
        for b in range(lo, hi):
            prob = H.Problem.dense(N, M, seed=3000 + b)
            prob.c.nthreads = 1
            r = (H.solve_reference if use_ref else H.solve_oracle)(prob, "dense", max_iterations=100)
            acc += r.ncalls - 1
        return acc
    t0 = time.perf_counter()
    with cf.ThreadPoolExecutor(nthreads) as ex:
        per = max(1, nsample // nthreads)
        done = sum(ex.map(lambda k: work(k * per, (k + 1) * per), range(nthreads)))
    return done, time.perf_counter() - t0, use_ref


def cpu_dense_sample(H, N, M, iterations):
    """One dense solve of a reduced C5 problem (N x M) through the reference (rank-1 J'J + dpptrf),
    capped at `iterations`; returns (iterations done, seconds without the callback, is_reference)."""
    use_ref = H.reference_lib() is not None
    prob = H.Problem.dense(N, M, seed=5)
    prob.c.nthreads = 0
    t0 = time.perf_counter()
    r = (H.solve_reference if use_ref else H.solve_oracle)(prob, "dense", max_iterations=iterations)
    dt = time.perf_counter() - t0 - r.cb_seconds
    return max(r.ncalls - 1, 1), dt, use_ref


def reference_line(args, val, t_total, cfg, cpu):
    return {"impl": "reference", "metric": "dogleg_iterations_per_sec", "value": val, "unit": "iterations/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * t_total / max(args.steps, 1), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": cfg, "cpu_baseline": cpu,
            "e2e": {"value": val, "unit": "iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}


def reference_arm(args, rank, world, dist):
    """The reference's own CPU implementation (unmodified dogleg.c from oracle/_ref; its CHOLMOD
    calls are served by the oracle's restatement because SuiteSparse is not installable here) on
    the same config; each step is a bounded sample: one solve capped at a few iterations."""
    if rank != 0:
        return
    from support import harness as H
    if args.config == "c3":
        nthreads = os.cpu_count() or 1
        nsample = 200 * nthreads
        args.steps, args.warmup = min(args.steps, 3), min(args.warmup, 1)
        it_total = t_total = 0.0
        for s in range(args.warmup + args.steps):
            done, dt, use_ref = cpu_batched_sample(H, 16, 256, nsample, nthreads)
            if s >= args.warmup:
                it_total += done
                t_total += dt
        val = it_total / t_total
        cpu = {"value": val, "unit": "iterations/s", "cores": nthreads, "kind": "reference" if use_ref else "port",
               "sample": f"{nsample} problems of the batch per step through dogleg_optimize_dense2 on {nthreads} threads "
                         "(problem construction and callback included)"}
        print(json.dumps(reference_line(args, val, t_total, {"workload": f"batched dense (c3): {args.batch} independent problems, "
                                                             "Nstate=16, Nmeas=256"}, cpu)), flush=True)
        return
    if args.config == "c5":
        args.steps, args.warmup = min(args.steps, 2), 0
        Ns, Ms = 1024, 4096
        it_total = t_total = 0.0
        for s in range(args.steps):
            done, dt, use_ref = cpu_dense_sample(H, Ns, Ms, args.ref_iterations)
            it_total += done
            t_total += dt
        val = it_total / t_total
        cpu = {"value": val, "unit": "iterations/s", "cores": 1, "kind": "reference" if use_ref else "port",
               "sample": f"REDUCED problem Nstate={Ns}, Nmeas={Ms} (the full {args.c5_states} x {args.c5_rows} J'J needs "
                         "~40 min per evaluation on one core: 4.2e12 FMA at the measured 1.7 GFMA/s), solve capped at "
                         f"{args.ref_iterations} iterations"}
        print(json.dumps(reference_line(args, val, t_total, {"workload": f"large dense (c5): Nstate={args.c5_states}, "
                                                             f"Nmeas={args.c5_rows}", "sampled_as": f"Nstate={Ns}, Nmeas={Ms}"},
                                        cpu)), flush=True)
        return
    # the reference is a single-threaded scalar code: the bundle-adjustment config is sampled at 1/10 scale
    ref_cfg = "c4m" if args.config == "c4" else args.config
    prob = make_problem(H, ref_cfg)
    prob.c.nthreads = 0
    use_ref = H.reference_lib() is not None
    solve = H.solve_reference if use_ref else H.solve_oracle
    cap = args.ref_iterations
    t_total, it_total, t_analyze = 0.0, 0, 0.0
    args.steps = min(args.steps, 5)        # each reference step costs seconds of CPU time
    args.warmup = min(args.warmup, 1)
    RL = H.reference_lib()
    if use_ref:
        RL.orc_shim_analyze_seconds.restype = C.c_double
        RL.orc_shim_analyze_seconds.argtypes = [C.c_int]
    for s in range(args.warmup + args.steps):
        if use_ref:
            RL.orc_shim_analyze_seconds(1)
        t0 = time.perf_counter()
        r = solve(prob, "sparse", max_iterations=cap)
        dt = time.perf_counter() - t0 - r.cb_seconds
        iters = r.ncalls - 1 if r.accepted < 0 else r.accepted     # no rejections on this problem: evaluations-1
        if s >= args.warmup:
            t_total += dt
            it_total += max(iters, 1)
            t_analyze += float(RL.orc_shim_analyze_seconds(1)) if use_ref else 0.0
    val = it_total / t_total
    line = {"impl": "reference", "metric": "dogleg_iterations_per_sec", "value": val, "unit": "iterations/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * t_total / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(args.config), "Nstate": prob.N, "Nmeas": prob.M, "NJnnz": prob.nnz,
                       "callback_time": "excluded",
                       "sampled_as": None if ref_cfg == args.config else workload_name(ref_cfg)},
            "cpu_baseline": {"value": val, "unit": "iterations/s", "cores": 1,
                             "kind": "reference" if use_ref else "port",
                             "value_excl_symbolic_analysis": it_total / max(t_total - t_analyze, 1e-9),
                             "symbolic_analysis_s_per_step": t_analyze / max(args.steps, 1),
                             "sample": f"full problem, solve capped at {cap} iterations per step (the reference repeats its "
                                       "symbolic analysis in every solve, so the cap inflates its share); CHOLMOD served by "
                                       "oracle/cholmod_shim.c (simplicial LDL' restatement, SuiteSparse unavailable)"},
            "e2e": {"value": val, "unit": "iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def workload_name(cfg):
    c = CONFIGS[cfg]
    if c[0] == "ba":
        return (f"synthetic bundle adjustment ({cfg}): {c[1]} cameras x {c[2]} points, {c[3]} observations/point, "
                f"camera window {c[4]}, {c[5]} permille long-range observations")
    ncam, nframes, npts = c
    return f"mrcal-shaped sparse calibration ({cfg}): {ncam} cams x {nframes} frames x {npts} points"


def dump_outputs(args, **arrays):
    """--dump-outputs: what the last timed step returned to its caller, one DIR/<name>.npy per array (float64),
    so that two builds can be compared output for output on identical, seeded inputs."""
    if not args.dump_outputs:
        return
    os.makedirs(args.dump_outputs, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(args.dump_outputs, name + ".npy"), np.asarray(a, dtype=np.float64))


def bench_c3(args, rank, world, local, dist, brief=False):
    """Config C3: B independent dense problems (Nstate=16, Nmeas=256), split evenly over the GPUs
    (strong scaling, no data-path collective). One step = the whole batch solved once."""
    import torch
    import libdogleg_b200 as dlb
    from support import harness as H
    L = dlb.load()
    L.dogleg_gpu_set_device(local)
    torch.cuda.set_device(local)
    N, M, Btot = 16, 256, args.batch
    B = Btot // world
    DL = H.dev_problems_lib()
    p0 = np.zeros((B, N))
    dev = DL.dlb_dev_problem_create_batched(B, M, N, 3000 + rank * B, H.as_dp(p0))
    assert dev
    st = np.zeros(8)

    def solve():
        rc, p, n2, it = H.solve_batched(dev, p0, N, M, max_iterations=100)
        assert rc == B
        L.dogleg_gpu_batched_stats(H.as_dp(st))
        return it, st.copy(), p, n2
    for _ in range(args.warmup):
        solve()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    sampler = ClockSampler(local)
    sampler.start()
    sampler.wait_first()
    steps = min(args.steps, 20) if brief else args.steps
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    t0 = time.perf_counter()
    iters = launches = 0
    k_ms = cb_ms = trials = 0.0
    for _ in range(steps):
        it_each, s, p_last, n2_last = solve()
        it = int(it_each.sum())
        iters += it
        launches += int(s[0])
        trials += s[1]
        k_ms += s[2]
        cb_ms += s[3]
    e1.record()
    torch.cuda.synchronize()
    wall = max(time.perf_counter() - t0, e0.elapsed_time(e1) * 1e-3)
    clocks = sampler.finish()
    t_all = barrier_max(dist, wall)
    iters_all = barrier_sum(dist, iters)
    peak, how = peaks()
    alg_per_trial = 8 * (M * N + M)                      # SURVEY.md 8(d): bytes one problem-trial must read
    ach = trials * alg_per_trial / (k_ms * 1e-3) / 1e9
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        # the reference's dense path, one solve per problem, on every host core (it is re-entrant
        # through the ...2 entry points with vnlog off); bounded sample of the same batch
        nthreads = os.cpu_count() or 1
        nsample = 400 * nthreads
        done, dt, use_ref = cpu_batched_sample(H, N, M, nsample, nthreads)
        cpu = {"value": done / dt, "unit": "iterations/s", "cores": nthreads, "kind": "reference" if use_ref else "port",
               "sample": f"first {nsample} problems of the batch through the reference's dogleg_optimize_dense2, "
                         f"{nthreads} threads (problem construction and callback included; evaluations-1 counted)"}
    line = None
    if rank == 0:
        line = {"metric": "dogleg_iterations_per_sec", "value": iters_all / t_all, "unit": "iterations/s",
                "n_gpus": world, "steps": steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_all / steps,
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": f"batched dense (c3): {Btot} independent problems, Nstate=16, Nmeas=256",
                           "problems_per_gpu": B, "iterations_per_problem": iters / steps / B,
                           "trials_per_step": trials / steps, "callback": "device model kernel, included in the time",
                           "l2_policy": f"{B * (M * N + M) * 8 / 1e6:.0f} MB per trial exceeds the 126 MB L2",
                           "parallelism": f"batch split over {world} GPU(s), no communication"},
                "clocks": clocks, "gpu_launches": launches,
                "e2e": {"value": iters_all / t_all, "unit": "iterations/s",
                        "h2d_bytes_per_step": B * N * 8, "d2h_bytes_per_step": B * (N * 8 + 12),
                        "note": "same call: start points from pageable host memory in, solutions out; the Jacobians "
                                "are produced on the device by the callback (a host-Jacobian batched API does not exist)"},
                "roofline": {"bound": "hbm", "kernel": "k_batched_trial", "achieved": ach, "peak": peak,
                             "peak_source": how, "unit": "GB/s", "frac": ach / peak,
                             "traffic": (measured_traffic("c3", "k_batched_trial_per_problem_trial") or 0) * trials / max(launches, 1)
                             if N == 16 and M == 256 and measured_traffic("c3", "k_batched_trial_per_problem_trial") else None,
                             "algorithmic_bytes_per_launch": alg_per_trial * trials / max(launches, 1),
                             "avg_launch_ms": k_ms / max(launches, 1), "callback_ms_per_launch": cb_ms / max(launches, 1)},
                "cpu_baseline": cpu}
        if not brief:
            dump_outputs(args, p=p_last, norm2x=n2_last, iterations=it_each)
    DL.dlb_dev_problem_free(dev)
    L.dogleg_gpu_release_cache()
    return line if rank == 0 else None


_dgemm_peak = []


def measure_dgemm_peak():
    """FP64 matrix-multiply peak of this GPU, measured with cuBLAS DGEMM (torch.matmul, 8192^3):
    the denominator for the DMMA kernels; MEASURED_PEAKS.json has no FP64 figure."""
    import torch
    if _dgemm_peak:
        return _dgemm_peak[0]
    n = 8192
    a = torch.randn(n, n, dtype=torch.float64, device="cuda")
    b = torch.randn(n, n, dtype=torch.float64, device="cuda")
    torch.matmul(a, b)
    torch.cuda.synchronize()
    best = 1e9
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        torch.matmul(a, b)
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1) * 1e-3)
    del a, b
    torch.cuda.empty_cache()
    _dgemm_peak.append(2.0 * n ** 3 / best / 1e12)
    return _dgemm_peak[0]


def bench_c5(args, rank, world, local, dist, brief=False):
    """Config C5: one large dense problem (Nstate=4096, Nmeas=500k by default), Jacobian produced on
    the device; J'J on the DMMA SYRK kernel, blocked DMMA Cholesky. N > 1: the rows of J are split
    evenly over the ranks (dogleg_gpu_optimize_dense_sharded): every rank forms the J'J of its rows,
    the partial N x N fronts / gradients / |Jv|^2 are summed with ncclAllReduce, strong scaling."""
    import torch
    import libdogleg_b200 as dlb
    from support import harness as H
    L = dlb.load()
    L.dogleg_gpu_set_device(local)
    torch.cuda.set_device(local)
    N, M = args.c5_states, args.c5_rows
    DL = H.dev_problems_lib()
    p0 = np.zeros((1, N))
    sharded = world > 1
    row_b, row_e = H.shard_columns(M, world, 1)[rank] if sharded else (0, M)
    if sharded:
        if not getattr(args, "_nccl_ready", False):
            nccl_setup(L, rank, world, dist)
            args._nccl_ready = True
        DL.dlb_dev_problem_create_dense_slice.restype = C.c_void_p
        DL.dlb_dev_problem_create_dense_slice.argtypes = [C.c_int, C.c_int, C.c_int, C.c_ulonglong, H.dp]
        dev = DL.dlb_dev_problem_create_dense_slice(row_b, row_e - row_b, N, 5, H.as_dp(p0))
        L.dogleg_gpu_optimize_dense_sharded.restype = C.c_double
        L.dogleg_gpu_optimize_dense_sharded.argtypes = [H.dp, C.c_uint, C.c_uint, C.c_uint, C.c_uint, C.c_void_p, C.c_void_p,
                                                        C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]
    else:
        dev = DL.dlb_dev_problem_create_batched(1, M, N, 5, H.as_dp(p0))       # A, b generated on the device
    assert dev
    P = H.make_params(L, max_iterations=args.c5_iterations)
    st = np.zeros(8)
    ph = np.zeros(8)

    def solve():
        p = p0[0].copy()
        if sharded:
            r = L.dogleg_gpu_optimize_dense_sharded(H.as_dp(p), N, M, row_b, row_e - row_b, None, DL.dlb_dev_cb_dense_ptr(),
                                                    C.c_void_p(dev), C.cast(C.byref(P), C.c_void_p), None)
        else:
            r = L.dogleg_gpu_optimize_dense(H.as_dp(p), N, M, DL.dlb_dev_cb_dense_ptr(), C.c_void_p(dev), C.byref(P), None)
        assert r >= 0, L.dogleg_gpu_last_error()
        L.dogleg_gpu_get_stats(None, H.as_dp(st))
        return r, st.copy(), p
    warmup = min(args.warmup, 1) if brief else args.warmup
    for _ in range(warmup):
        solve()
    steps = min(args.steps, 3) if brief else args.steps
    if dist is not None:
        dist.barrier()
    sampler = ClockSampler(local)
    sampler.start()
    sampler.wait_first()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    t0 = time.perf_counter()
    iters = launches = 0
    for _ in range(steps):
        cost, s, p_last = solve()
        iters += int(s[0])
        launches += int(s[4])
    e1.record()
    torch.cuda.synchronize()
    wall = max(time.perf_counter() - t0, e0.elapsed_time(e1) * 1e-3)
    if dist is not None:
        dist.barrier()
    clocks = sampler.finish()
    wall = barrier_max(dist, wall)
    launches = int(barrier_sum(dist, launches))
    # per-phase device time of one more solve (events around every phase)
    os.environ["DOGLEG_GPU_PHASE_TIMING"] = "1"
    _, s, _ = solve()
    os.environ["DOGLEG_GPU_PHASE_TIMING"] = "0"
    L.dogleg_gpu_get_phase_ms(H.as_dp(ph))
    if rank != 0:
        DL.dlb_dev_problem_free(dev)
        L.dogleg_gpu_release_cache()
        return None
    nfact, nevals = max(s[3], 1), max(s[1], 1)
    syrk_ms = ph[3] / nfact
    flops = float(row_e - row_b) * N * (N + 1)           # SURVEY.md 8(d): triangle of J'J, this rank's rows
    dgemm = measure_dgemm_peak()
    ach = flops / (syrk_ms * 1e-3) / 1e12
    names = ["h2d", "gradient", "cauchy_Jv", "assemble_syrk", "factor", "solve", "step_Jv", "d2h_p"]
    line = {"metric": "dogleg_iterations_per_sec", "value": iters / wall, "unit": "iterations/s", "n_gpus": world,
            "steps": steps, "warmup": warmup, "ms_per_step": 1e3 * wall / steps, "higher_is_better": True,
            "scaling": "weak" if world == 1 else "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"large dense (c5): Nstate={N}, Nmeas={M}", "iterations_per_solve": iters / steps,
                       "final_cost": cost, "callback": "device model kernel, included",
                       "parallelism": "single GPU" if world == 1 else
                       f"rows of J split over {world} GPUs, ncclAllReduce of the partial J'J / gradient / |Jv|^2, Cholesky replicated",
                       "l2_policy": f"J is {M * N * 8 / 1e9:.1f} GB, far beyond the 126 MB L2"},
            "clocks": clocks, "gpu_launches": launches,
            "e2e": {"value": iters / wall, "unit": "iterations/s", "h2d_bytes_per_step": N * 8, "d2h_bytes_per_step": N * 8 + 8,
                    "note": "device-callback solve through dogleg_gpu_optimize_dense; a host-callback solve would move "
                            f"{M * N * 8 / 1e9:.1f} GB over PCIe per evaluation"},
            "roofline": {"bound": "tensor", "kernel": "k_dense_syrk_dmma", "achieved": ach, "peak": dgemm,
                         "peak_source": "cuBLAS DGEMM 8192^3 measured in this run", "unit": "TFLOP/s", "frac": ach / dgemm,
                         "traffic": measured_traffic("c5", "k_dense_syrk_dmma") if (N, M, world) == (4096, 500000, 1) else None,
                         "flops_per_launch": flops, "avg_launch_ms": syrk_ms,
                         "all_phases_ms_per_call": {n: round(float(v) / (nfact if i in (3, 4, 5) else nevals), 4)
                                                    for i, (n, v) in enumerate(zip(names, ph))}},
            "cpu_baseline": None}
    if world == 1 and not args.no_cpu_baseline:
        Ns, Ms = 1024, 4096
        done, dt, use_ref = cpu_dense_sample(H, Ns, Ms, args.ref_iterations)
        line["cpu_baseline"] = {"value": done / dt, "unit": "iterations/s", "cores": 1, "kind": "reference" if use_ref else "port",
                                "sample": f"REDUCED problem Nstate={Ns}, Nmeas={Ms} through the reference's dense path (rank-1 J'J + "
                                          f"dpptrf), capped at {args.ref_iterations} iterations; at full size one evaluation needs "
                                          "~40 min on one core (4.2e12 FMA at the measured 1.7 GFMA/s)"}
    if not brief:
        dump_outputs(args, p=p_last, norm2x=[cost])
    DL.dlb_dev_problem_free(dev)
    L.dogleg_gpu_release_cache()
    return line


def bench_sparse(args, cfg, rank, world, local, dist, brief=False, mode=None):
    """One sparse config (c2 / c4 families) through the public API; returns the JSON line (rank 0) or None.
    brief: the short form used for `extra_configs` (fewer steps, no parity run, bounded CPU sample).
    mode (N>1): "sharded" = ONE problem row-sharded over the ranks (strong scaling), "replicas" = every rank
    solves the whole problem by itself at the same time, no communication (weak scaling)."""
    import torch
    import libdogleg_b200 as dlb
    from libdogleg_b200 import ffi
    from support import harness as H
    L = dlb.load()
    if L.dogleg_gpu_device_count() <= 0:
        raise SystemExit("bench.py: no CUDA device (libdogleg-b200 has no CPU fallback)")
    L.dogleg_gpu_set_device(local)
    torch.cuda.set_device(local)
    L.dogleg_gpu_assume_pattern_unchanged.argtypes = [C.c_int]
    L.dogleg_gpu_assume_pattern_unchanged.restype = None
    ba = CONFIGS[cfg][0] == "ba"
    steps = args.steps if not brief else (3 if ba else min(args.steps, 20))
    warmup = args.warmup if not brief else (1 if ba else min(args.warmup, 3))

    t0 = time.perf_counter()
    prob = make_problem(H, cfg)                          # the same global problem on every rank
    Jp, Ji = prob.pattern()
    t_problem = time.perf_counter() - t0
    N, M, nnz = prob.N, prob.M, prob.nnz
    PL = H.problems_lib()
    DL = H.dev_problems_lib()
    P = H.make_params(L, max_iterations=100)
    st = np.zeros(8)
    if mode is None:
        mode = "sharded" if world > 1 else "single"
    sharded = world > 1 and mode == "sharded"
    replicas = world > 1 and not sharded
    if sharded:
        if not getattr(args, "_nccl_ready", False):
            nccl_setup(L, rank, world, dist)
            args._nccl_ready = True
        L.dogleg_gpu_optimize_sparse_sharded.restype = C.c_double
        L.dogleg_gpu_optimize_sparse_sharded.argtypes = [H.dp, C.c_uint, C.c_uint, H.ip, H.ip, C.c_uint, C.c_uint,
                                                         C.c_void_p, C.c_void_p, C.c_void_p,
                                                         C.POINTER(ffi.Parameters), C.POINTER(C.c_void_p)]
        col_b, col_e = H.shard_columns(M, world, shard_alignment(cfg))[rank]   # whole frames / points per rank
        lprob = prob.slice(col_b, col_e - col_b)
    else:
        col_b, col_e, lprob = 0, M, prob
    dev = DL.dlb_dev_problem_create(C.cast(lprob.ptr, C.c_void_p))
    assert dev, "device problem upload failed"
    if world > 1:
        lprob.c.nthreads = max(1, (os.cpu_count() or 1) // world)     # the host callbacks of all ranks share the cores

    def solve_device():
        p = prob.p0()
        if sharded:
            r = L.dogleg_gpu_optimize_sparse_sharded(H.as_dp(p), N, M, H.as_ip(Jp), H.as_ip(Ji), col_b, col_e - col_b,
                                                     None, DL.dlb_dev_cb_sparse_ptr(), C.c_void_p(dev), C.byref(P), None)
        else:
            r = L.dogleg_gpu_optimize_sparse(H.as_dp(p), N, M, nnz, H.as_ip(Jp), H.as_ip(Ji),
                                             DL.dlb_dev_cb_sparse_ptr(), C.c_void_p(dev), C.byref(P), None)
        assert r >= 0, L.dogleg_gpu_last_error()
        L.dogleg_gpu_get_stats(None, H.as_dp(st))
        return r, st.copy(), p

    def solve_host():
        p = prob.p0()
        lprob.reset()
        lprob.trace(False)
        if sharded:
            r = L.dogleg_gpu_optimize_sparse_sharded(H.as_dp(p), N, M, H.as_ip(Jp), H.as_ip(Ji), col_b, col_e - col_b,
                                                     PL.dlb_cb_sparse_ptr(), None, C.cast(lprob.ptr, C.c_void_p),
                                                     C.byref(P), None)
        else:
            r = L.dogleg_optimize2(H.as_dp(p), N, M, nnz, PL.dlb_cb_sparse_ptr(), C.cast(prob.ptr, C.c_void_p),
                                   C.byref(P), None)
        assert r >= 0, L.dogleg_gpu_last_error()
        L.dogleg_gpu_get_stats(None, H.as_dp(st))
        return r, st.copy(), lprob.c.cb_seconds, p

    # ---------------- the first solve: symbolic analysis + index upload (then served by the engine cache) ----
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    solve_device()
    torch.cuda.synchronize()
    t_first = time.perf_counter() - t0
    # the cost of the default (safe) reuse check: a hash of the whole pattern once per solve
    L.dogleg_gpu_assume_pattern_unchanged(0)
    t0 = time.perf_counter()
    if not args.profile_only:
        solve_device()
    torch.cuda.synchronize()
    t_checked = time.perf_counter() - t0
    # the benchmark passes the same arrays every time and says so: sample comparison only
    L.dogleg_gpu_assume_pattern_unchanged(1)

    # ---------------- value: device-resident inputs ----------------
    for _ in range(warmup):
        solve_device()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    sampler = ClockSampler(local)
    sampler.start()
    sampler.wait_first()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    t0 = time.perf_counter()
    iters = launches = 0
    cost = p_dev = None
    for _ in range(steps):
        cost, s, p_dev = solve_device()
        iters += int(s[0])
        launches += int(s[4])
    e1.record()
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    dev_s = e0.elapsed_time(e1) * 1e-3
    if dist is not None:
        dist.barrier()
    clocks = sampler.finish()
    t_value = barrier_max(dist, max(wall, dev_s))
    # sharded: one global problem, every rank walks the same iterations; replicas: every rank its own solve
    iters_all = int(barrier_sum(dist, iters)) if replicas else iters
    launches = int(barrier_sum(dist, launches))
    value = iters_all / t_value
    # the callback's share: CUDA events around the model kernel, one extra solve
    DL.dlb_dev_problem_timing.argtypes = [C.c_void_p, C.c_int]
    DL.dlb_dev_problem_ms.restype = C.c_double
    DL.dlb_dev_problem_ms.argtypes = [C.c_void_p]
    DL.dlb_dev_problem_timing(C.c_void_p(dev), 1)
    s_cb = s
    if not args.profile_only:
        _, s_cb, _ = solve_device()
    cb_ms = float(DL.dlb_dev_problem_ms(C.c_void_p(dev)))
    DL.dlb_dev_problem_timing(C.c_void_p(dev), 0)
    cb_ms_all = barrier_max(dist, cb_ms)
    per_solve_ms = 1e3 * t_value / max(steps, 1)
    value_excl_cb = iters_all / max(steps, 1) / max(1e-9, (per_solve_ms - cb_ms_all) * 1e-3)

    # ---------------- e2e: host callbacks, pinned H2D inside the timed region ----------------
    e2e = None
    p_host = cost_host = None
    if not args.profile_only:
        # plain callbacks first (everything is copied after the callback returns), then the same callback
        # announcing its progress (dogleg_gpu_host_progress): the pinned H2D overlaps the callback
        solve_host()
        if dist is not None:
            dist.barrier()
        t_plain, it_plain = 0.0, 0
        def lib_seconds(dt, cbs):
            # sharded: the ranks meet in a collective after every evaluation, so the slowest rank's callback is on
            # everybody's critical path: subtract the largest callback time, from the largest wall time
            return barrier_max(dist, dt) - barrier_max(dist, cbs) if sharded else dt - cbs
        for _ in range(2 if ba else 3):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            _, s, cbs, _ = solve_host()
            torch.cuda.synchronize()
            t_plain += lib_seconds(time.perf_counter() - t0, cbs)
            it_plain += int(s[0])
        t_plain = barrier_max(dist, t_plain)
        if replicas:
            it_plain = int(barrier_sum(dist, it_plain))
        lprob.c.progress = C.cast(L.dogleg_gpu_host_progress, C.c_void_p).value
        for _ in range(1):
            solve_host()
        if dist is not None:
            dist.barrier()
        t_lib = 0.0
        it2 = 0
        h2d = d2h = 0.0
        e2e_steps = (2 if ba else max(3, min(steps, 20)))
        for _ in range(e2e_steps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            cost_host, s, cbs, p_host = solve_host()
            torch.cuda.synchronize()
            t_lib += lib_seconds(time.perf_counter() - t0, cbs)
            it2 += int(s[0])
            h2d += s[5]
            d2h += s[6]
        t_e2e = barrier_max(dist, t_lib)
        if replicas:
            it2 = int(barrier_sum(dist, it2))
        h2d, d2h = barrier_sum(dist, h2d), barrier_sum(dist, d2h)
        lprob.c.progress = None
        e2e = {"value": it2 / t_e2e, "unit": "iterations/s",
               "h2d_bytes_per_step": h2d / e2e_steps, "d2h_bytes_per_step": d2h / e2e_steps, "steps": e2e_steps,
               "value_plain_callback": it_plain / t_plain,
               "note": "dogleg_optimize2 with host callbacks writing into the library's pinned buffers; all copies are inside the "
                       "timed region, the time spent inside the callback body is subtracted (it is user code, identical for "
                       "the reference arm). `value`: the callback fills its outputs front to back and announces progress "
                       "(dogleg_gpu_host_progress), so the side-stream H2D overlaps the callback and only the tail is exposed; "
                       "`value_plain_callback`: the same callback without announcements (all of the H2D after it returns)"
                       + ("; row-sharded: per solve the largest callback time over the ranks is subtracted from the largest "
                          "wall time (the ranks meet in a collective after every evaluation)" if sharded else "")}

    # ---------------- roofline: per-phase device time of the engine calls dogleg_optimize* issues ----------------
    roof = None
    if rank == 0:
        E = H.Engine(ffi.SOLVE_SPARSE, N, M, nnz)
        x, Jx = prob.evaluate(prob.p0())
        E.load_sparse(0, prob.p0(), x, Jp, Ji, Jx)
        fused = False
        E.evaluate(0)
        fused = E.has_trial()
        if fused:
            E.trial(0, 1, 1e9)
        else:
            E.cauchy(0)
            E.factorize(0, 0.0)
            E.gauss_newton(0)
            E.step(0, 1, ffi.STEP_GAUSSNEWTON, 1e9)
        reps = 1 if args.profile_only else (10 if not ba else 3)
        L.dlb_engine_enable_timing(E.h, 1)
        for _ in range(reps):
            L.dlb_engine_evaluate(E.h, 0, 0, 0.0)      # device-resident: no H2D; a fresh point: nothing cached
            if fused:
                E.trial(0, 1, 1e9)
            else:
                E.cauchy(0)
                E.factorize(0, 0.0)
                E.gauss_newton(0)
                E.step(0, 1, ffi.STEP_GAUSSNEWTON, 1e9)
        ph = np.zeros(8)
        L.dlb_engine_phase_ms(E.h, H.as_dp(ph))
        ph /= reps
        if fused:
            names = ["h2d", "evaluation_pass", "-", "evaluation_reduce", "trial_kernel", "-", "-", "d2h_p"]
        elif L.dlb_engine_has_fused_eval(E.h):
            # fused evaluation, per-operation trial step (trees with fronts beyond shared memory: bundle adjustment)
            names = ["h2d", "evaluation_pass", "cauchy_Jv", "evaluation_reduce", "factor", "solve", "step_Jv", "d2h_p"]
        else:
            names = ["h2d", "gradient", "cauchy_Jv", "assemble", "factor", "solve", "step_Jv", "d2h_p"]
        phases = {n: round(float(v), 5) for n, v in zip(names, ph) if n != "-"}
        info = (C.c_longlong * 8)()
        L.dlb_symbolic_info(L.dlb_engine_symbolic(E.h), info)
        nnzL, flops = int(info[3]), float(info[6])
        nnzA = int(np.count_nonzero(np.tril(E.JtJ(0, 0.0)))) if N <= 4096 else None
        peak, how = peaks()
        total_ms = float(sum(ph))
        if fused:
            # SURVEY.md 8(d), "fused gradient+assembly": 12 nnz + 4 (M+1) + 8 M + 8 N + 8 nnzA bytes per pass
            alg = 12 * nnz + 4 * (M + 1) + 8 * M + 8 * N + 8 * (nnzA or 0)
            dur = ph[1] * 1e-3
            ach = alg / dur / 1e9
            roof = {"bound": "hbm", "kernel": "k_sparse_assemble<grad> (fused evaluation: Jt*x, |x|^2 and the class blocks of "
                                              "Jt*Jt' in one pass over Jt)",
                    "achieved": ach, "peak": peak, "peak_source": how, "unit": "GB/s", "frac": ach / peak,
                    "traffic": measured_traffic(cfg, "k_sparse_assemble_grad"),
                    "algorithmic_bytes_per_launch": alg,
                    "algorithmic_bytes_formula": "12*NJnnz + 4*(Nmeas+1) + 8*Nmeas + 8*Nstate + 8*nnz(tril JtJ)",
                    "nnz_tril_JtJ": nnzA, "avg_launch_ms": dur * 1e3, "all_phases_ms": phases, "nnzL": nnzL,
                    "device_time_share": {n: round(float(v) / total_ms, 3) for n, v in zip(names, ph) if n != "-" and v > 0},
                    # the phase with the largest share of the library's device time: one cooperative launch for
                    # Cauchy + factorization + solves + step + expected improvement; a chain of small dependent
                    # steps (6 grid barriers), bound by latency -- both roofline fractions are stated for the record
                    "dominant_phase": {"name": "k_trial (whole trial step in one persistent kernel)", "bound": "latency",
                                       "avg_launch_ms": float(ph[4]), "share_of_device_time": float(ph[4]) / total_ms,
                                       "factor_flops": flops, "bytes_8_nnzA_plus_nnzL": 8 * ((nnzA or 0) + nnzL),
                                       "frac_of_hbm_peak": 8 * ((nnzA or 0) + nnzL) / (ph[4] * 1e-3) / 1e9 / peak if ph[4] > 0 else None,
                                       "tflops": flops / (ph[4] * 1e-3) / 1e12 if ph[4] > 0 else None}}
        else:
            jv_bytes = 12 * nnz + 4 * (M + 1) + 8 * N if ba else 8 * (nnzA or 0) + 8 * N
            fe = "evaluation_pass" in names
            if fe:
                # the evaluation = pass + per-state reduction: quoted together against the gradient's algorithmic bytes
                algs = {"evaluation_pass": 12 * nnz + 4 * (M + 1) + 8 * M + 8 * N, "cauchy_Jv": jv_bytes, "step_Jv": jv_bytes}
                durs = {"evaluation_pass": ph[1] + ph[3], "cauchy_Jv": ph[2], "step_Jv": ph[6]}
            else:
                algs = {"gradient": 12 * nnz + 4 * (M + 1) + 8 * M + 8 * N, "cauchy_Jv": jv_bytes, "step_Jv": jv_bytes,
                        "assemble": 12 * nnz + 4 * (M + 1) + 8 * (nnzA or 0)}
                durs = {k: ph[names.index(k)] for k in algs}
            top = max(algs, key=lambda k: durs[k])
            dur = durs[top] * 1e-3
            ach = algs[top] / dur / 1e9
            kname = {"gradient": "k_sparse_grad_small(+reduce)" if ba else "k_range_grad(+reduce)",
                     "evaluation_pass": "k_sparse_grad_small + k_sparse_assemble_small + k_sparse_grad_reduce (the whole evaluation)",
                     "cauchy_Jv": "k_sparse_jv_small(+sum)" if ba else "k_gpart_quadform",
                     "step_Jv": "k_step_apply + " + ("k_sparse_jv_small(+sum)" if ba else "k_gpart_quadform"),
                     "assemble": "k_sparse_assemble" + ("_small" if ba else "")}[top]
            stream = {"kernel": kname, "achieved_GBs": ach, "frac_of_hbm": ach / peak, "algorithmic_bytes_per_launch": algs[top],
                      "avg_launch_ms": dur * 1e3, "traffic": measured_traffic(cfg, kname)}
            fdur = ph[names.index("factor")] * 1e-3
            if fdur > dur:
                # the numeric factorization dominates (bundle adjustment): quote it against the FP64 tensor bound,
                # SURVEY.md 8(d): sum_j colcount_j^2 flops, >= 8 (nnzA + nnzL) bytes
                dg = measure_dgemm_peak()
                roof = {"bound": "tensor", "kernel": "multifrontal factorization (k_leaf_fronts_mma, k_extend_gather, k_front_level, "
                                                    "k_bf_step / k_bf_diag + k_bf_trsm, k_bf_gemm)",
                        "achieved": flops / fdur / 1e12, "peak": dg, "peak_source": "cuBLAS DGEMM 8192^3 measured in this run",
                        "unit": "TFLOP/s", "frac": flops / fdur / 1e12 / dg, "traffic": None, "flops_per_launch": flops,
                        "avg_launch_ms": fdur * 1e3, "all_phases_ms": phases, "nnzL": nnzL,
                        "front_storage_doubles": int(info[5]), "levels": int(info[2]),
                        "device_time_share": {n: round(float(v) / total_ms, 3) for n, v in zip(names, ph) if v > 0},
                        "solve_GBs": (16 * nnzL + 32 * N) / (ph[names.index("solve")] * 1e-3) / 1e9,
                        "solve_frac_of_hbm": (16 * nnzL + 32 * N) / (ph[names.index("solve")] * 1e-3) / 1e9 / peak,
                        "streaming_kernel": stream}
            else:
                roof = {"bound": "hbm", "kernel": kname, "achieved": ach, "peak": peak, "peak_source": how, "unit": "GB/s",
                        "frac": ach / peak, "traffic": stream["traffic"], "algorithmic_bytes_per_launch": algs[top],
                        "avg_launch_ms": dur * 1e3, "all_phases_ms": phases, "nnzL": nnzL}
        E.close()

    # ---------------- CPU baseline + parity: the reference on this box's host cores ----------------
    cpu = parity = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline and not args.profile_only and not (brief and ba):
        use_ref = H.reference_lib() is not None
        solve = H.solve_reference if use_ref else H.solve_oracle
        ref_cfg = "c4m" if cfg == "c4" else cfg
        rprob = prob if ref_cfg == cfg else make_problem(H, ref_cfg)
        full = (not brief) and rprob is prob and N <= 4096           # C2: the reference converges in ~15 s
        RL = H.reference_lib()
        if use_ref:
            RL.orc_shim_analyze_seconds.restype = C.c_double
            RL.orc_shim_analyze_seconds.argtypes = [C.c_int]
            RL.orc_shim_analyze_seconds(1)
        t0 = time.perf_counter()
        r = solve(rprob, "sparse", max_iterations=100 if full else args.ref_iterations)
        dt = time.perf_counter() - t0 - r.cb_seconds
        t_an = float(RL.orc_shim_analyze_seconds(1)) if use_ref else 0.0
        its = max(r.ncalls - 1, 1)
        what = "same problem" if rprob is prob else workload_name(ref_cfg) + " (1/10 of the workload)"
        cpu = {"value": its / dt, "unit": "iterations/s", "cores": 1,
               "kind": "reference" if use_ref else "port",
               "value_excl_symbolic_analysis": its / max(dt - t_an, 1e-9), "symbolic_analysis_s": t_an,
               "sample": f"{what}, one solve " + ("run to convergence" if full else f"capped at {args.ref_iterations} iterations")
                         + "; unmodified reference dogleg.c, CHOLMOD calls served by oracle/cholmod_shim.c (SuiteSparse "
                           "not installable here); the reference repeats cholmod_analyze in every solve"}
        if full:
            # the reference solved the same problem to convergence: compare what the GPU arms returned
            def cmp(pg, cg):
                return {"cost_rel_err": abs(cg - r.norm2x) / abs(r.norm2x),
                        "p_max_abs_err": float(np.max(np.abs(pg - r.p))),
                        "p_max_abs_err_over_max_abs_p": float(np.max(np.abs(pg - r.p)) / max(1.0, np.max(np.abs(r.p))))}
            parity = {"reference": "oracle/_ref (unmodified dogleg.c) solved to convergence on the same inputs",
                      "reference_evaluations": int(r.ncalls), "reference_cost": r.norm2x,
                      "device_callbacks": dict(cmp(p_dev, cost), evaluations=int(s_cb[1]),
                                               evaluations_equal=int(s_cb[1]) == int(r.ncalls)),
                      "tolerance": {"cost_rel": 1e-9, "p": 1e-7}}
            if p_host is not None:
                parity["host_callbacks"] = dict(cmp(p_host, cost_host), evaluations=int(s[1]),
                                                evaluations_equal=int(s[1]) == int(r.ncalls))

    line = None
    if rank == 0:
        gather = sharded and N >= 16384
        line = {"metric": "dogleg_iterations_per_sec", "value": value, "unit": "iterations/s",
                "n_gpus": world, "steps": steps, "warmup": warmup,
                "ms_per_step": per_solve_ms, "higher_is_better": True,
                "scaling": "strong" if sharded else "weak",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": workload_name(cfg), "Nstate": N, "Nmeas": M, "NJnnz": nnz,
                           "iterations_per_solve": iters / max(steps, 1), "final_cost": cost,
                           "parallelism": "single GPU" if world == 1 else
                           (f"{world} independent solves of this problem at the same time, one per GPU, no communication "
                            f"(the row-sharded solve of ONE problem over the {world} GPUs is reported under `sharded`)") if replicas else
                           (f"measurement columns split by points over {world} GPUs; the ranks exchange their slices of x / Jt values "
                            "(grouped ncclBroadcast), everything downstream replicated" if gather else
                            f"measurements row-sharded by frames over {world} GPUs, one grouped ncclAllReduce of [class blocks | "
                            "Jt*x | |x|^2] per evaluation, everything after it (quadratic forms, factorization, step) rank-local"),
                           "l2_policy": f"inputs ({8 * nnz / 1e6:.0f} MB of Jacobian values per evaluation) "
                                        + ("exceed" if 8 * nnz > 126e6 else "DO NOT exceed") + " the 126 MB L2",
                           "step": "one full solve through the public API: context creation, engine-cache HIT (device/pinned buffers "
                                   "and the symbolic analysis of the first solve are reused; the caller declares the pattern "
                                   "unchanged, so only a sample of it is compared), all iterations, result download",
                           "engine_cache": "hit", "first_solve_s": t_first,
                           "first_solve_note": "includes the symbolic analysis, index build and upload (once per pattern)",
                           "solve_with_full_pattern_hash_ms": 1e3 * t_checked,
                           "problem_generation_s": t_problem},
                "value_excl_callback": value_excl_cb, "callback_ms_per_solve": cb_ms_all,
                "callback_note": "the synthetic model kernel (tests/support/problems_dev.cu) is user code on the solver's stream; "
                                 "`value` includes it",
                "clocks": clocks, "e2e": e2e, "gpu_launches": launches, "roofline": roof, "cpu_baseline": cpu}
        if parity is not None:
            line["parity"] = parity
        if not brief:
            dump_outputs(args, p=p_dev, norm2x=[cost])
        if sharded:
            cs = np.zeros(2)
            L.dogleg_gpu_get_comm_stats(H.as_dp(cs))
            line["comm"] = {"collectives_per_solve": float(cs[0]), "bytes_per_rank_per_solve": float(cs[1]),
                            "evaluations_per_solve": float(s_cb[1]),
                            "note": "grouped NCCL operations of the last timed solve on rank 0 (dogleg_gpu_get_comm_stats)"}
    DL.dlb_dev_problem_free(dev)
    L.dogleg_gpu_release_cache()
    return line


def trim_extra(line):
    """what `extra_configs` keeps of a config's own line"""
    if line is None:
        return None
    keep = ("value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "config", "clocks", "e2e",
            "gpu_launches", "roofline", "cpu_baseline", "value_excl_callback")
    return {k: line[k] for k in keep if k in line}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default=None, choices=list(CONFIGS) + ["c3", "c5"])
    ap.add_argument("--extras", default="default", choices=["default", "all", "none"],
                    help="without --config: which other configs ride along in `extra_configs` "
                         "(default: c3, c5 and -- on one GPU -- c4; all: c4 sharded as well)")
    ap.add_argument("--c5-states", type=int, default=4096)
    ap.add_argument("--c5-rows", type=int, default=500000)
    ap.add_argument("--c5-iterations", type=int, default=3)
    ap.add_argument("--batch", type=int, default=100000, help="c3: number of problems in the whole job")
    ap.add_argument("--ref-iterations", type=int, default=2)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--profile-only", action="store_true", help="short run for ncu: no e2e, no cpu baseline")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step of the headline config returned (final p, cost; c3: per "
                         "problem, iterations too) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.steps < 1:
        ap.error("--dump-outputs needs at least one timed step")
    rank, world, local, dist = dist_setup(args.gpus)
    headline = args.config or "c2"
    if args.config is None:
        args.config = "c2"

    if args.impl == "reference":
        reference_arm(args, rank, world, dist)
        if dist is not None:
            dist.barrier()
            dist.destroy_process_group()
        return

    def run(cfg, brief):
        if cfg == "c3":
            return bench_c3(args, rank, world, local, dist, brief=brief)
        if cfg == "c5":
            return bench_c5(args, rank, world, local, dist, brief=brief)
        if world > 1 and CONFIGS[cfg][0] != "ba":
            # a C2-sized iteration (0.4 ms, half of it a dependency chain that does not shard) gains nothing from being
            # split: the whole-job throughput of N GPUs is N solves at a time; the sharded solve rides along
            line = bench_sparse(args, cfg, rank, world, local, dist, brief=brief, mode="replicas")
            sh = bench_sparse(args, cfg, rank, world, local, dist, brief=True, mode="sharded")
            if rank == 0 and line is not None and sh is not None:
                line["sharded"] = {k: sh[k] for k in ("value", "unit", "scaling", "ms_per_step", "value_excl_callback", "e2e",
                                                      "gpu_launches", "comm") if k in sh}
                line["sharded"]["parallelism"] = sh["config"]["parallelism"]
                line["sharded"]["final_cost"] = sh["config"]["final_cost"]
            return line
        return bench_sparse(args, cfg, rank, world, local, dist, brief=brief)

    line = run(headline, False)
    extras = {}
    single = not any(a.startswith("--config") for a in sys.argv[1:])
    if single and args.extras != "none" and not args.profile_only:
        todo = ["c3", "c5"] + (["c4"] if (world == 1 or args.extras == "all") else [])
        saved = (args.steps, args.warmup)
        for cfg in todo:
            t0 = time.perf_counter()
            try:
                ex = trim_extra(run(cfg, True))
            except Exception as exc:                   # an extra must never cost the headline line
                ex = {"error": f"{type(exc).__name__}: {exc}"[:400]} if rank == 0 else None
            if rank == 0 and ex is not None:
                ex["wall_s"] = round(time.perf_counter() - t0, 1)
                extras[cfg] = ex
            args.steps, args.warmup = saved
    if rank == 0 and line is not None:
        if extras:
            line["extra_configs"] = extras
        print(json.dumps(line), flush=True)
    if getattr(args, "_nccl_ready", False):
        import libdogleg_b200 as dlb
        dlb.load().dogleg_gpu_nccl_finalize()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
