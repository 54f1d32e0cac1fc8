"""The final state of a batched solve (dogleg_gpu_batch_t) at C3's shape: B = 100 000, Nstate = 16, Nmeas = 256.

1. What a handle costs the solve: dogleg_gpu_optimize_dense_batched2 with and without returnBatch, alternating
   on the same device-generated batch after a warm-up solve of each. Wall time per solve (host clock around
   whole solves, which end in a device synchronise) and k_batched_trial ms per launch (CUDA events, from
   dogleg_gpu_batched_stats). The difference is the final J'J stores plus the device-to-device copy into the
   handle.
2. k_batched_factor through dogleg_gpu_batch_covariance_device (full and packed) and
   dogleg_gpu_batch_solve_device (nrhs = 1 and 16): CUDA events around --reps launches after a warm-up launch.
   The handle's J'J alone is 205 MB, more than the 126 MB L2, so every launch reads it from HBM. Each time is
   reported beside the bytes the call must move and that traffic over the time as a fraction of the 7.7 TB/s
   HBM figure of the HGX B200 data sheet.
3. With --compare-tree DIR (another checkout of this repository, built): `bench.py --config c3 --dump-outputs`
   alternately from this tree and from DIR, --bench-rounds times each. Reports whether the dumped p, cost and
   iteration files are identical and the trial-kernel ms per launch of every run, so that the difference
   between the trees can be set against the spread of repeated runs of the same tree.

Reads the GPU's name and power limit in the same run. Prints one JSON document (and writes it to --out).
Run from the repository root after build():  python profiles/micro/batched_results.py --out FILE
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

HBM_DATASHEET_GBS = 7700.0          # NVIDIA HGX B200 data sheet, per GPU (the figure DESIGN.md section 4 uses)


def gpu_identity():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as ex:                  # pragma: no cover - reported, not hidden
        return {"error": str(ex)}


def solve(H, L, dev, p0, N, M, handle, max_iterations):
    P = H.make_params(L, max_iterations=max_iterations)
    p = p0.copy()
    B = p.shape[0]
    n2 = np.zeros(B)
    it = np.zeros(B, dtype=np.int32)
    h = C.c_void_p()
    st = np.zeros(8)
    t0 = time.perf_counter()
    rc = L.dogleg_gpu_optimize_dense_batched2(H.as_dp(p), N, M, B, H.dev_problems_lib().dlb_dev_cb_dense_batched_ptr(),
                                              C.c_void_p(dev), C.byref(P), H.as_dp(n2), H.as_ip(it),
                                              C.byref(h) if handle else None)
    wall = time.perf_counter() - t0
    assert rc == B, L.dogleg_gpu_last_error()
    L.dogleg_gpu_batched_stats(H.as_dp(st))
    return {"wall_ms": 1e3 * wall, "kernel_ms_per_launch": st[2] / st[0], "launches": int(st[0])}, (p, n2, it), h


def time_calls(torch, call, reps):
    call()                                              # warm-up: module load, shared-memory attribute
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        call()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def bench_c3(tree, outdir):
    out = subprocess.run([sys.executable, "bench.py", "--config", "c3", "--gpus", "1", "--steps", "5", "--warmup", "1",
                          "--no-cpu-baseline", "--dump-outputs", outdir], cwd=tree, capture_output=True, text=True)
    if out.returncode != 0:
        raise RuntimeError(f"bench.py in {tree} failed:\n{out.stderr[-3000:]}")
    line = json.loads([s for s in out.stdout.splitlines() if s.startswith("{")][-1])
    return {"value": line["value"], "avg_launch_ms": line["roofline"]["avg_launch_ms"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=100000)
    ap.add_argument("--rounds", type=int, default=3, help="alternating solves with / without a handle after the warm-up")
    ap.add_argument("--reps", type=int, default=50, help="timed launches per k_batched_factor variant")
    ap.add_argument("--max-iterations", type=int, default=100)
    ap.add_argument("--compare-tree", default=None, help="a built checkout to compare bench.py --config c3 against")
    ap.add_argument("--compare-label", default="other", help="what --compare-tree is, for the report")
    ap.add_argument("--bench-rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    import libdogleg_b200 as dlb
    from support import harness as H
    L = dlb.load()
    if L.dogleg_gpu_device_count() <= 0:
        raise SystemExit("no CUDA device: this measurement needs the GPU")
    DL = H.dev_problems_lib()
    doc = {"gpu": gpu_identity(), "hbm_peak_used_GBs": HBM_DATASHEET_GBS,
           "hbm_peak_source": "NVIDIA HGX B200 data sheet, per GPU (not a measured peak)"}

    # ---- 1. the solve with and without a handle ----
    N, M, B = 16, 256, args.batch
    p0 = np.zeros((B, N))
    dev = DL.dlb_dev_problem_create_batched(B, M, N, 3000, H.as_dp(p0))
    assert dev
    runs = {False: [], True: []}
    outs = {}
    for handle in (False, True):                         # warm-up: module load, workspace allocation
        _, _, h = solve(H, L, dev, p0, N, M, handle, args.max_iterations)
        if handle:
            L.dogleg_gpu_batch_free(C.byref(h))
    for _ in range(args.rounds):
        for handle in (False, True):
            r, o, h = solve(H, L, dev, p0, N, M, handle, args.max_iterations)
            runs[handle].append(r)
            outs[handle] = o
            if handle:
                L.dogleg_gpu_batch_free(C.byref(h))
    _, _, h = solve(H, L, dev, p0, N, M, True, args.max_iterations)          # the handle timed below
    DL.dlb_dev_problem_free(dev)
    L.dogleg_gpu_release_batched_cache()

    def summary(rs):
        return {"wall_ms_each": [round(r["wall_ms"], 2) for r in rs],
                "kernel_ms_per_launch_each": [round(r["kernel_ms_per_launch"], 4) for r in rs],
                "launches": rs[0]["launches"]}
    w0 = np.mean([r["wall_ms"] for r in runs[False]])
    w1 = np.mean([r["wall_ms"] for r in runs[True]])
    doc["solve_with_handle"] = {
        "B": B, "Nstate": N, "Nmeas": M, "max_iterations": args.max_iterations,
        "without": summary(runs[False]), "with": summary(runs[True]),
        "extra_wall_ms_per_solve": w1 - w0,
        "handle_bytes": B * (N * N * 8 + 8 + 4),
        "outputs_identical": all(np.array_equal(u, v) for u, v in zip(outs[False], outs[True]))}

    # ---- 2. k_batched_factor ----
    stream = torch.cuda.current_stream().cuda_stream
    jtj_bytes = B * N * N * 8 + B * 8 * 2              # J'J in, lambda in and out
    res = {}
    for packed in (False, True):
        n_out = N * (N + 1) // 2 if packed else N * N
        d_out = torch.empty((B, n_out), dtype=torch.float64, device="cuda")
        ms = time_calls(torch, lambda: L.dogleg_gpu_batch_covariance_device(h, d_out.data_ptr(), int(packed), stream),
                        args.reps)
        nbytes = jtj_bytes + B * n_out * 8
        res["covariance_packed" if packed else "covariance_full"] = {
            "ms": ms, "bytes": nbytes, "GBs": nbytes / (ms * 1e-3) / 1e9,
            "fraction_of_datasheet_hbm": nbytes / (ms * 1e-3) / 1e9 / HBM_DATASHEET_GBS}
    for nrhs in (1, 16):
        d_R = torch.randn((B, nrhs, N), dtype=torch.float64, device="cuda")
        d_X = torch.empty_like(d_R)
        ms = time_calls(torch, lambda: L.dogleg_gpu_batch_solve_device(h, d_R.data_ptr(), d_X.data_ptr(), nrhs, stream),
                        args.reps)
        nbytes = jtj_bytes + 2 * B * nrhs * N * 8
        res[f"solve_nrhs{nrhs}"] = {"ms": ms, "bytes": nbytes, "GBs": nbytes / (ms * 1e-3) / 1e9,
                                    "fraction_of_datasheet_hbm": nbytes / (ms * 1e-3) / 1e9 / HBM_DATASHEET_GBS}
    L.dogleg_gpu_batch_free(C.byref(h))
    doc["k_batched_factor"] = dict(res, reps=args.reps, l2_note="205 MB of J'J per launch exceeds the 126 MB L2")

    # ---- 3. bench.py --config c3 against another tree ----
    if args.compare_tree:
        trees = {"this": ROOT, "other": os.path.abspath(args.compare_tree)}
        bench = {"this": [], "other": []}
        identical = True
        with tempfile.TemporaryDirectory() as td:
            for r in range(args.bench_rounds):
                for name, tree in trees.items():
                    d = os.path.join(td, f"{name}{r}")
                    bench[name].append(bench_c3(tree, d))
                for f in ("p.npy", "norm2x.npy", "iterations.npy"):
                    a = np.load(os.path.join(td, f"this{r}", f))
                    b = np.load(os.path.join(td, f"other{r}", f))
                    identical &= bool(np.array_equal(a, b))
        ms = {k: [round(x["avg_launch_ms"], 4) for x in v] for k, v in bench.items()}
        doc["bench_c3_against_other_tree"] = {
            "other_tree": args.compare_label,
            "outputs_identical_every_round": identical,
            "trial_kernel_ms_per_launch": ms,
            "spread_within_this": max(ms["this"]) - min(ms["this"]),
            "spread_within_other": max(ms["other"]) - min(ms["other"]),
            "iterations_per_s": {k: [round(x["value"]) for x in v] for k, v in bench.items()}}

    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
