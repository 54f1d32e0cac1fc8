"""Ragged batched dense solves (dogleg_gpu_optimize_dense_batched_ragged) against the uniform form on the same batch
zero-padded to its longest problem. Test model of tests/support/ragged_dev.cu (problem b = the first Nmeas[b] rows of
k_gen_batched's problem seed + b); both forms use the same callback code.

(a) C3's shape, every count 256 (B = 100 000, Nstate = 16): ragged against uniform, trial-kernel ms per launch over a
    full solve, iteration counts and outputs compared.
(b) B = 100 000, Nstate = 16, counts drawn (seed 0) log-uniform on [16, 1024]: the ragged form (longest-first order),
    the same with the identity order (--identity-lib: a scratch build of libdogleg.so that skips the sort), and the
    uniform form padded to the longest count. For each: ms per trial launch at the initial point (max_iterations = 0:
    one launch, every problem active) and over a full solve, the algorithmic bytes of that first launch
    (sum over problems of 8 (M_b N + M_b)) over its time as a share of the 7.7 TB/s data-sheet figure, the x + J
    workspace bytes, the end-to-end solve time, and whether p, cost and iterations are identical.
(c) Outlierness factors (featureSize 1) on (b)'s batch at the returned p: the ragged device form against the uniform
    one on the padded data, CUDA events over --reps launches after a warm-up launch.

Every shape is warmed up before it is timed. The per-problem data (3.1 GB ragged, 13 GB padded at (b)) are far over
the 126 MB L2, so every launch streams from HBM. Reads the GPU's name and power limit in the same run.
Run from the repository root after build():  python profiles/micro/batched_ragged.py --out FILE
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
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from batched_results import HBM_DATASHEET_GBS, gpu_identity, time_calls  # noqa: E402

N = 16


def skewed_counts(B):
    rng = np.random.default_rng(0)
    return np.floor(np.exp(rng.uniform(np.log(16), np.log(1024), B))).astype(np.uint32)


def run(HR, L, H, dev, p0, counts, ragged, max_iterations):
    """One solve; (stats dict, (p, n2, it))."""
    t0 = time.perf_counter()
    if ragged:
        rc, p, n2, it, _ = HR.solve(dev, p0, N, counts, max_iterations=max_iterations)
    else:
        rc, p, n2, it, _ = HR.solve_padded(dev, p0, N, max_iterations=max_iterations)
    wall = time.perf_counter() - t0
    assert rc == len(counts)
    st = np.zeros(8)
    L.dogleg_gpu_batched_stats(H.as_dp(st))
    return {"wall_ms": 1e3 * wall, "kernel_ms_per_launch": st[2] / st[0], "launches": int(st[0]),
            "callback_ms": st[3]}, (p, n2, it)


def measure(HR, L, H, dev, p0, counts, ragged, max_iterations, rounds):
    """Warm-up, then `rounds` first-launch timings and `rounds` full solves."""
    run(HR, L, H, dev, p0, counts, ragged, 0)
    first = [run(HR, L, H, dev, p0, counts, ragged, 0)[0]["kernel_ms_per_launch"] for _ in range(rounds)]
    full = [run(HR, L, H, dev, p0, counts, ragged, max_iterations) for _ in range(rounds)]
    return {"first_launch_ms": first, "full": [f[0] for f in full]}, full[-1][1]


def only_ragged(args):
    """--only-ragged (the child process of --identity-lib): (b)'s ragged solve with the library at --lib."""
    from libdogleg_b200 import ffi
    if args.lib:
        ffi.lib_path = lambda: args.lib
    from support import harness as H
    from support import ragged as HR
    L = ffi.load()
    counts = skewed_counts(args.batch)
    dev, p0 = HR.create(counts, N, 5000)
    r, (p, n2, it) = measure(HR, L, H, dev, p0, counts, True, args.max_iterations, args.rounds)
    HR.free(dev)
    np.savez(args.only_ragged, p=p, n2=n2, it=it)
    print(json.dumps(r))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=100000)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=20, help="timed outlierness launches per form")
    ap.add_argument("--max-iterations", type=int, default=100)
    ap.add_argument("--identity-lib", default=None, help="a libdogleg.so built to take the problems in index order")
    ap.add_argument("--lib", default=None, help=argparse.SUPPRESS)
    ap.add_argument("--only-ragged", default=None, help=argparse.SUPPRESS)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.only_ragged:
        return only_ragged(args)

    import torch
    import libdogleg_b200 as dlb
    from support import harness as H
    from support import ragged as HR
    L = dlb.load()
    if L.dogleg_gpu_device_count() <= 0:
        raise SystemExit("no CUDA device: this measurement needs the GPU")
    doc = {"gpu": gpu_identity(), "hbm_peak_used_GBs": HBM_DATASHEET_GBS,
           "hbm_peak_source": "NVIDIA HGX B200 data sheet, per GPU (not a measured peak)"}
    B = args.batch

    # ---- (a) C3's shape, all counts 256 ----
    counts = np.full(B, 256, dtype=np.uint32)
    dev, p0 = HR.create(counts, N, 3000)
    a = {}
    outs = {}
    for ragged in (True, False):
        run(HR, L, H, dev, p0, counts, ragged, 0)                               # warm-up of both shapes
    for _ in range(2):
        for ragged in (True, False):
            r, o = run(HR, L, H, dev, p0, counts, ragged, args.max_iterations)
            a.setdefault("ragged" if ragged else "uniform", []).append(r)
            outs[ragged] = o
    HR.free(dev)
    L.dogleg_gpu_release_batched_cache()
    a["outputs_identical"] = all(np.array_equal(u, v) for u, v in zip(outs[True], outs[False]))
    a["iterations_equal"] = bool(np.array_equal(outs[True][2], outs[False][2]))
    doc["a_c3_all_256"] = a

    # ---- (b) the skewed batch ----
    counts = skewed_counts(B)
    dev, p0 = HR.create(counts, N, 5000)
    Mpad = HR.mpad(dev)
    rows = int(HR.offsets(counts)[-1])
    bytes_first = 8.0 * rows * (N + 1)                                          # every problem active
    bb = {"counts": {"mean": float(counts.mean()), "min": int(counts.min()), "max": int(counts.max()), "rows": rows},
          "padded_to": Mpad, "algorithmic_bytes_first_launch": {"ragged": bytes_first, "padded": bytes_first},
          "streamed_bytes_first_launch_padded": 8.0 * B * Mpad * (N + 1),
          "workspace_xJ_bytes": {"ragged": 8.0 * rows * (N + 1) + 8.0 * (B + 1) + 4.0 * B,
                                 "padded": 8.0 * B * Mpad * (N + 1)}}
    res = {}
    res["ragged"], o_r = measure(HR, L, H, dev, p0, counts, True, args.max_iterations, args.rounds)
    res["padded"], o_p = measure(HR, L, H, dev, p0, counts, False, args.max_iterations, args.rounds)
    bb["outputs_identical_ragged_padded"] = all(np.array_equal(u, v) for u, v in zip(o_r, o_p))
    if args.identity_lib:
        L.dogleg_gpu_release_batched_cache()
        with tempfile.TemporaryDirectory() as tmp:
            f = os.path.join(tmp, "identity.npz")
            out = subprocess.run([sys.executable, os.path.abspath(__file__), "--only-ragged", f, "--lib", args.identity_lib,
                                  "--batch", str(B), "--rounds", str(args.rounds), "--max-iterations",
                                  str(args.max_iterations)], capture_output=True, text=True)
            if out.returncode != 0:
                raise RuntimeError(out.stderr[-3000:])
            res["ragged_identity_order"] = json.loads(out.stdout.strip().splitlines()[-1])
            z = np.load(f)
            bb["outputs_identical_ragged_identity"] = all(np.array_equal(u, z[k]) for u, k in zip(o_r, ("p", "n2", "it")))
        res["ragged_again"], _ = measure(HR, L, H, dev, p0, counts, True, args.max_iterations, args.rounds)
    for k, r in res.items():
        ms = min(r["first_launch_ms"])
        r["first_launch_share_of_7p7TBs"] = bytes_first / (ms * 1e-3) / (HBM_DATASHEET_GBS * 1e9)
    bb["runs"] = res

    # ---- (c) outlierness on (b)'s batch at the returned p ----
    p = o_r[0]
    off = HR.offsets(counts)
    d_p = torch.from_numpy(p).cuda()
    d_off = torch.from_numpy(off).cuda()
    d_x = torch.empty(rows, dtype=torch.float64, device="cuda")
    d_J = torch.empty((rows, N), dtype=torch.float64, device="cuda")
    d_xp = torch.empty((B, Mpad), dtype=torch.float64, device="cuda")
    d_Jp = torch.empty((B, Mpad, N), dtype=torch.float64, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    torch.cuda.synchronize()
    HR.lib().dlb_ragged_cb(d_p.data_ptr(), d_x.data_ptr(), d_J.data_ptr(), d_off.data_ptr(), None, B, stream, dev)
    HR.lib().dlb_ragged_cb_padded(d_p.data_ptr(), d_xp.data_ptr(), d_Jp.data_ptr(), None, B, stream, dev)
    torch.cuda.synchronize()
    rr, _, _, _, hr = HR.solve(dev, p0, N, counts, handle=True, max_iterations=args.max_iterations)
    rp, _, _, _, hp = HR.solve_padded(dev, p0, N, handle=True, max_iterations=args.max_iterations)
    HR.free(dev)
    L.dogleg_gpu_release_batched_cache()
    d_scale = torch.ones(B, dtype=torch.float64, device="cuda")               # kept: the factors are comparable
    d_f = torch.full((rows,), float("nan"), dtype=torch.float64, device="cuda")
    d_fp = torch.full((B, Mpad), float("nan"), dtype=torch.float64, device="cuda")
    ms_r = time_calls(torch, lambda: L.dogleg_gpu_batch_outlierness_ragged_device(
        hr, d_x.data_ptr(), d_J.data_ptr(), 1, None, None, d_scale.data_ptr(), d_f.data_ptr(), stream), args.reps)
    ms_p = time_calls(torch, lambda: L.dogleg_gpu_batch_outlierness_device(
        hp, d_xp.data_ptr(), d_Jp.data_ptr(), Mpad, 1, Mpad, None, d_scale.data_ptr(), d_fp.data_ptr(), stream), args.reps)
    fr, fp = d_f.cpu().numpy(), d_fp.cpu().numpy()
    same = all(np.array_equal(fr[off[b]:off[b + 1]], fp[b, :counts[b]]) for b in range(0, B, 97))
    ob = 8.0 * rows * (N + 1)
    doc["c_outlierness_fs1"] = {"ragged_ms": ms_r, "padded_ms": ms_p, "algorithmic_bytes": ob,
                                "ragged_share_of_7p7TBs": ob / (ms_r * 1e-3) / (HBM_DATASHEET_GBS * 1e9),
                                "padded_streamed_bytes": 8.0 * B * Mpad * (N + 1),
                                "factors_identical_every_97th_problem": bool(same),
                                "note": "input scales 1 (kept), so that both forms compute the same factors"}
    L.dogleg_gpu_batch_free(C.byref(hr))
    L.dogleg_gpu_batch_free(C.byref(hp))
    doc["b_skewed"] = bb
    text = json.dumps(doc, indent=2)
    print(text)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
