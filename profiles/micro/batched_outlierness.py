"""k_batched_outlierness (dogleg_gpu_batch_outlierness_device) at C3's shape: B = 100 000, Nstate = 16, Nmeas = 256.

1. A dense batched solve with a handle (test model, seeds 3000 + b). x and J at the returned p come from the test
   model's device callback (dlb_dev_cb_dense_batched, every problem active).
2. For featureSize 1 and 2: the kernel time from CUDA events around --reps launches after a warm-up launch, the
   bytes it must move (J alone is 3.28 GB, far over the 126 MB L2, so every launch streams it from HBM) and that
   traffic over the time as a fraction of the 7.7 TB/s HBM figure of the HGX B200 data sheet.
3. For comparison, in the same process: k_batched_trial at the initial point of a solve with max_iterations = 0 (one
   launch that streams the same J and stops before the step), the trial kernel's mean per launch over the full
   solve of step 1, and dogleg_gpu_batch_covariance_device (k_batched_factor).
4. A numpy spot check of --spot random problems: J* inv(JtJ + lambda I) J*' and the reference's formula.
5. With --compare-tree DIR (another built checkout): bench.py --config c3 --dump-outputs alternately from both trees
   (profiles/micro/batched_results.py does the runs); reports whether p, cost and iterations are identical.

Reads the GPU's name and power limit in the same run. Prints one JSON document (and writes it to --out).
Run from the repository root after build():  python profiles/micro/batched_outlierness.py --out FILE
"""
import argparse
import ctypes as C
import json
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from batched_results import HBM_DATASHEET_GBS, bench_c3, gpu_identity, solve, time_calls  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=100000)
    ap.add_argument("--reps", type=int, default=50, help="timed launches per variant")
    ap.add_argument("--max-iterations", type=int, default=100)
    ap.add_argument("--spot", type=int, default=100, help="problems checked against numpy")
    ap.add_argument("--compare-tree", default=None, help="a built checkout to compare bench.py --config c3 against")
    ap.add_argument("--compare-label", default="other", help="what --compare-tree is, for the report")
    ap.add_argument("--bench-rounds", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    import libdogleg_b200 as dlb
    from support import harness as H
    from test_gpu_batched_outlierness import dense_xJ, numpy_outlierness
    L = dlb.load()
    if L.dogleg_gpu_device_count() <= 0:
        raise SystemExit("no CUDA device: this measurement needs the GPU")
    DL = H.dev_problems_lib()
    DL.dlb_dev_cb_dense_batched.argtypes = [C.c_void_p] * 4 + [C.c_int, C.c_void_p, C.c_void_p]
    DL.dlb_dev_cb_dense_batched.restype = None
    doc = {"gpu": gpu_identity(), "hbm_peak_used_GBs": HBM_DATASHEET_GBS,
           "hbm_peak_source": "NVIDIA HGX B200 data sheet, per GPU (not a measured peak)"}

    # ---- 1. the solve, x and J at the returned p ----
    N, M, B, seed = 16, 256, args.batch, 3000
    p0 = np.zeros((B, N))
    dev = DL.dlb_dev_problem_create_batched(B, M, N, seed, H.as_dp(p0))
    assert dev
    solve(H, L, dev, p0, N, M, False, 0)                             # warm-up: module load, workspace
    first = [solve(H, L, dev, p0, N, M, False, 0)[0]["kernel_ms_per_launch"] for _ in range(5)]
    full, (p, n2, it), h = solve(H, L, dev, p0, N, M, True, args.max_iterations)
    stream = torch.cuda.current_stream().cuda_stream
    d_p = torch.from_numpy(p).cuda()
    d_x = torch.empty((B, M), dtype=torch.float64, device="cuda")
    d_J = torch.empty((B, M, N), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    DL.dlb_dev_cb_dense_batched(d_p.data_ptr(), d_x.data_ptr(), d_J.data_ptr(), None, B, stream, dev)
    torch.cuda.synchronize()
    DL.dlb_dev_problem_free(dev)
    L.dogleg_gpu_release_batched_cache()
    st = np.zeros(B, dtype=np.int32)
    lam = np.zeros(B)
    assert L.dogleg_gpu_batch_status(h, H.as_ip(st), H.as_dp(lam)) == 0

    # ---- 2. k_batched_outlierness ----
    res = {}
    outs = {}
    for fs in (1, 2):
        nfeat = M // fs
        d_scale = torch.full((B,), -1.0, dtype=torch.float64, device="cuda")
        d_f = torch.empty((B, nfeat), dtype=torch.float64, device="cuda")

        def call():
            d_scale.fill_(-1.0)
            assert L.dogleg_gpu_batch_outlierness_device(h, d_x.data_ptr(), d_J.data_ptr(), M, fs, nfeat, None,
                                                         d_scale.data_ptr(), d_f.data_ptr(), stream) == 0
        call()
        torch.cuda.synchronize()
        outs[fs] = (d_f.cpu().numpy(), d_scale.cpu().numpy())

        def kernel_only():
            assert L.dogleg_gpu_batch_outlierness_device(h, d_x.data_ptr(), d_J.data_ptr(), M, fs, nfeat, None,
                                                         d_scale.data_ptr(), d_f.data_ptr(), stream) == 0
        ms = time_calls(torch, kernel_only, args.reps)
        by = {"J": B * M * N * 8, "x": B * M * 8, "JtJ": B * N * N * 8, "lambda_scale_in_out": B * 8 * 4,
              "factors": B * nfeat * 8}
        nbytes = sum(by.values())
        res[f"featureSize{fs}"] = {"ms": ms, "bytes": nbytes, "bytes_by_array": by, "GBs": nbytes / (ms * 1e-3) / 1e9,
                                   "fraction_of_datasheet_hbm": nbytes / (ms * 1e-3) / 1e9 / HBM_DATASHEET_GBS,
                                   "datasheet_bound_ms": nbytes / (HBM_DATASHEET_GBS * 1e9) * 1e3}
    doc["k_batched_outlierness"] = dict(res, B=B, Nstate=N, Nmeas=M, reps=args.reps,
                                        note="the timed launches keep the scale the first launch wrote; |x|^2 is "
                                             "summed in every launch all the same, so each does the whole work")

    # ---- 3. comparisons ----
    d_cov = torch.empty((B, N * N), dtype=torch.float64, device="cuda")
    cov_ms = time_calls(torch, lambda: L.dogleg_gpu_batch_covariance_device(h, d_cov.data_ptr(), 0, stream), args.reps)
    doc["compare"] = {
        "k_batched_trial_initial_point_ms_each": [round(x, 4) for x in first],
        "k_batched_trial_initial_point_note": "a solve with max_iterations = 0: one launch, every problem active, "
                                              "streams the same J and stops before the step",
        "k_batched_trial_full_solve_ms_per_launch": full["kernel_ms_per_launch"],
        "full_solve_launches": full["launches"],
        "covariance_full_ms": cov_ms}

    # ---- 4. numpy spot check ----
    rng = np.random.default_rng(11)
    worst = {1: 0.0, 2: 0.0}
    worst_scale = 0.0
    for b in rng.choice(B, size=min(args.spot, B), replace=False):
        x, J = dense_xJ(H, N, M, seed + int(b), p[b])
        for fs in (1, 2):
            fw, sw = numpy_outlierness(x, J, lam[b], fs, M // fs)
            f, sc = outs[fs][0][b], outs[fs][1][b]
            worst[fs] = max(worst[fs], float(np.max(np.abs(f - fw) / np.maximum(np.abs(fw), 1e-12 * np.max(np.abs(fw))))))
            worst_scale = max(worst_scale, float(abs(sc - sw) / abs(sw)))
    doc["numpy_spot_check"] = {"problems": min(args.spot, B), "max_rel_err_featureSize1": worst[1],
                               "max_rel_err_featureSize2": worst[2], "max_rel_err_scale": worst_scale,
                               "passed": bool(worst[1] <= 1e-7 and worst[2] <= 1e-7 and worst_scale <= 1e-9)}
    L.dogleg_gpu_batch_free(C.byref(h))

    # ---- 5. bench.py --config c3 against another tree ----
    if args.compare_tree:
        trees = {"this": ROOT, "other": os.path.abspath(args.compare_tree)}
        bench = {"this": [], "other": []}
        identical = True
        with tempfile.TemporaryDirectory() as td:
            for r in range(args.bench_rounds):
                for name, tree in trees.items():
                    bench[name].append(bench_c3(tree, os.path.join(td, f"{name}{r}")))
                for f in ("p.npy", "norm2x.npy", "iterations.npy"):
                    identical &= bool(np.array_equal(np.load(os.path.join(td, f"this{r}", f)),
                                                     np.load(os.path.join(td, f"other{r}", f))))
        doc["bench_c3_against_other_tree"] = {
            "other_tree": args.compare_label, "outputs_identical_every_round": identical,
            "trial_kernel_ms_per_launch": {k: [round(x["avg_launch_ms"], 4) for x in v] for k, v in bench.items()},
            "iterations_per_s": {k: [round(x["value"]) for x in v] for k, v in bench.items()}}

    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
