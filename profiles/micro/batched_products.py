"""Batched dense-products solves against the batched dense form, in one process.

1. C3's shape (B = 100 000, Nstate = 16, Nmeas = 256): dogleg_gpu_optimize_dense_batched and
   dogleg_gpu_optimize_dense_products_batched on the same device-generated batch, alternating, after a
   warm-up solve of each. Per form: iterations/s (host clock around whole solves, which end in a device
   synchronise), trials, k_batched_trial ms per launch and callback ms per launch (CUDA events, from
   dogleg_gpu_batched_stats), the bytes one problem-trial must read from HBM, and that traffic over the
   kernel time as a fraction of the 7.7 TB/s data-sheet figure.
2. A shape the dense form cannot hold (B = 40 000, Nstate = 16, Nmeas = 65 536: 336 GB of Jacobians) with
   the procedural callback, which regenerates every row on every evaluation.

Reads the GPU's name and power limit in the same run. Prints one JSON document (and writes it to --out).
Run from the repository root after build():  python profiles/micro/batched_products.py --out FILE
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

HBM_DATASHEET_GBS = 7700.0          # NVIDIA HGX B200 data sheet, per GPU


def gpu_identity():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as ex:                  # pragma: no cover - reported, not hidden
        return {"error": str(ex)}


def bytes_per_problem_trial(form, N, M):
    """Algorithmic HBM reads of one problem-trial in k_batched_trial (callback outputs only)."""
    if form == "dense":
        return 8 * (M * N + M)                         # J and x, streamed once
    return 8 * (N * (N + 1) // 2 + N + 1)              # packed upper J'J, J'x, |x|^2


def run_form(H, HP, L, form, dev, p0, N, M, packed, max_iterations):
    st = np.zeros(8)
    t0 = time.perf_counter()
    if form == "dense":
        rc, p, n2, it = H.solve_batched(dev, p0, N, M, max_iterations=max_iterations)
    else:
        rc, p, n2, it = HP.solve_batched(dev, p0, N, packed=packed, max_iterations=max_iterations)
    wall = time.perf_counter() - t0
    L.dogleg_gpu_batched_stats(H.as_dp(st))
    assert rc == p0.shape[0], rc
    return {"wall_s": wall, "iterations": int(it.sum()), "launches": int(st[0]), "trials": float(st[1]),
            "kernel_ms": float(st[2]), "callback_ms": float(st[3])}, (p, n2, it)


def summarise(runs, form, N, M):
    wall = sum(r["wall_s"] for r in runs)
    iters = sum(r["iterations"] for r in runs)
    launches = sum(r["launches"] for r in runs)
    trials = sum(r["trials"] for r in runs)
    k_ms = sum(r["kernel_ms"] for r in runs)
    cb_ms = sum(r["callback_ms"] for r in runs)
    bpt = bytes_per_problem_trial(form, N, M)
    gbs = trials * bpt / (k_ms * 1e-3) / 1e9
    return {"solves": len(runs), "iterations_per_s": iters / wall, "ms_per_solve": 1e3 * wall / len(runs),
            "ms_per_solve_each": [round(1e3 * r["wall_s"], 2) for r in runs],
            "trials_per_solve": trials / len(runs), "launches_per_solve": launches / len(runs),
            "kernel_ms_per_launch": k_ms / launches,
            "kernel_ms_per_launch_each": [round(r["kernel_ms"] / r["launches"], 4) for r in runs],
            "callback_ms_per_launch": cb_ms / launches,
            "algorithmic_bytes_per_problem_trial": bpt,
            "kernel_algorithmic_GBs": gbs, "kernel_hbm_fraction_of_datasheet": gbs / HBM_DATASHEET_GBS}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=100000)
    ap.add_argument("--rounds", type=int, default=3, help="alternating dense / products solves after the warm-up")
    ap.add_argument("--big-batch", type=int, default=40000)
    ap.add_argument("--big-meas", type=int, default=65536)
    ap.add_argument("--max-iterations", type=int, default=100)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import libdogleg_b200 as dlb
    from support import harness as H
    from support import products as HP
    L = dlb.load()
    if L.dogleg_gpu_device_count() <= 0:
        raise SystemExit("no CUDA device: this measurement needs the GPU")
    DL = H.dev_problems_lib()
    doc = {"gpu": gpu_identity(), "hbm_peak_used_GBs": HBM_DATASHEET_GBS}

    # ---- C3's shape, both forms, alternating ----
    N, M, B = 16, 256, args.batch
    p0 = np.zeros((B, N))
    dense = DL.dlb_dev_problem_create_batched(B, M, N, 3000, H.as_dp(p0))
    assert dense
    prod, p0p = HP.create_batched(B, M, N, 3000)          # the same seeds and generator code
    assert np.array_equal(p0, p0p)
    devs = {"dense": dense, "products": prod}
    runs = {"dense": [], "products": []}
    last = {}
    for form in runs:                                     # warm-up: module load, workspace allocation
        run_form(H, HP, L, form, devs[form], p0, N, M, True, args.max_iterations)
    for _ in range(args.rounds):
        for form in runs:
            r, out = run_form(H, HP, L, form, devs[form], p0, N, M, True, args.max_iterations)
            runs[form].append(r)
            last[form] = out
    DL.dlb_dev_problem_free(dense)
    HP.free(prod)
    L.dogleg_gpu_release_batched_cache()
    (pd, n2d, itd), (pp, n2p, itp) = last["dense"], last["products"]
    doc["c3_shape"] = {"B": B, "Nstate": N, "Nmeas": M, "products_layout": "packed upper",
                       "dense": summarise(runs["dense"], "dense", N, M),
                       "products": summarise(runs["products"], "products", N, M),
                       "forms_agree": {"equal_iterations": bool(np.array_equal(itd, itp)),
                                       "max_abs_dp": float(np.max(np.abs(pd - pp))),
                                       "max_rel_dnorm2x": float(np.max(np.abs(n2d - n2p) / n2d))}}

    # ---- beyond HBM: procedural callback, products form only ----
    Bb, Mb = args.big_batch, args.big_meas
    dev, p0 = HP.create_batched(Bb, Mb, N, 9000, stored=False)
    r, (p, n2, it) = run_form(H, HP, L, "products", dev, p0, N, Mb, True, args.max_iterations)
    HP.free(dev)
    L.dogleg_gpu_release_batched_cache()
    big = summarise([r], "products", N, Mb)
    big.update({"B": Bb, "Nstate": N, "Nmeas": Mb, "callback": "procedural (rows regenerated on every evaluation)",
                "dense_form_jacobian_GB": Bb * Mb * N * 8 / 1e9, "problems_finished": int(Bb),
                "iterations_per_problem": float(it.mean())})
    doc["beyond_hbm"] = big

    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
