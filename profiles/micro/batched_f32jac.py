"""Batched dense solves with a float Jacobian (dogleg_gpu_optimize_dense_batched_f32jac, _ragged_f32jac) against the
double form. Test model of tests/support/f32jac_dev.cu. The double form is driven by the widened twin callback
((double)(float)J), so both forms take the same steps, launch for launch, and differ only in the Jacobian's element type.

(a) C3's shape (B = 100 000, Nstate = 16, Nmeas = 256), full solve: per form, ms per trial launch
    (dogleg_gpu_batched_stats), callback ms per evaluation, end-to-end solve time, accepted steps per second, and the
    algorithmic bytes per launch (8M + 8MN per active problem for double J, 8M + 4MN for float J; the per-problem state
    is left out) over the kernel time as a share of the 7.7 TB/s data-sheet figure.
(b) C3's shape, first launch only (max_iterations = 0: one launch, every problem active), the bandwidth-bound case.
(c) The ragged measurement's skewed batch (B = 100 000, Nstate = 16, counts log-uniform on [16, 1024], seed 0), both
    ragged forms, full solve and first launch.
(d) Optionally bench.py --config c3 alternated with another built checkout (--compare-tree): dumped outputs compared.

The forms alternate within one process, --rounds times each, after a warm-up of every shape; the spread of the rounds
is reported beside the minimum. Per-problem data are 3.3 GB (C3) and 3.1 GB (skewed) of A alone, far over the 126 MB L2.
Reads the GPU's name and power limit in the same run.
Run from the repository root after build():  python profiles/micro/batched_f32jac.py --out FILE
"""
import argparse
import json
import os
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from batched_ragged import skewed_counts  # noqa: E402
from batched_results import HBM_DATASHEET_GBS, bench_c3, gpu_identity  # noqa: E402

N = 16
CALLBACK_NOTE = ("The test model (tests/support/f32jac_dev.cu) computes every value in double in both forms: per row it "
                 "reads N doubles of A, one double of b and the problem's p, and writes x as a double. The float callback "
                 "then stores each J entry rounded to float (4 bytes); the double form's callback (the widened twin) stores "
                 "the same rounded value as a double (8 bytes). A model that holds its inputs in float would read less; "
                 "these callback times are the test model's, not the library's.")


def run(HF, L, H, dev, p0, kind, counts, max_iterations):
    t0 = time.perf_counter()
    rc, p, n2, it, _ = HF.solve(kind, dev, p0, N, counts, max_iterations=max_iterations)
    wall = time.perf_counter() - t0
    assert rc == len(p0)
    st = np.zeros(8)
    L.dogleg_gpu_batched_stats(H.as_dp(st))
    return {"wall_ms": 1e3 * wall, "launches": int(st[0]), "active_problem_launches": st[1],
            "kernel_ms_per_launch": st[2] / st[0], "callback_ms_per_eval": st[3] / st[0],
            "accepted_steps": int(it.sum()), "accepted_steps_per_s": float(it.sum()) / wall}, (p, n2, it)


def per_problem_bytes(f32, m_rows):
    """Algorithmic bytes one launch streams for a problem of m_rows measurements: x and J."""
    return 8.0 * m_rows + (4.0 if f32 else 8.0) * m_rows * N


def summarise(runs, bytes_per_launch):
    ms = [r["kernel_ms_per_launch"] for r in runs]
    share = [b / (t * 1e-3) / (HBM_DATASHEET_GBS * 1e9) for b, t in zip(bytes_per_launch, ms)]
    return {"kernel_ms_per_launch": {"min": min(ms), "max": max(ms), "all": ms},
            "callback_ms_per_eval": [r["callback_ms_per_eval"] for r in runs],
            "solve_wall_ms": [r["wall_ms"] for r in runs],
            "accepted_steps_per_s": [r["accepted_steps_per_s"] for r in runs],
            "launches": runs[-1]["launches"], "accepted_steps": runs[-1]["accepted_steps"],
            "algorithmic_bytes_per_launch": bytes_per_launch[-1],
            "share_of_7p7TBs": {"at_min_ms": max(share), "all": share}}


def compare(HF, L, H, dev, p0, kinds, counts, max_iterations, rounds, bytes_fn):
    """Alternate the forms `rounds` times after a warm-up; returns {kind: summary} and whether the outputs agree."""
    for k in kinds:
        run(HF, L, H, dev, p0, k, counts, max_iterations)
    runs = {k: [] for k in kinds}
    outs = {}
    for _ in range(rounds):
        for k in kinds:
            r, o = run(HF, L, H, dev, p0, k, counts, max_iterations)
            runs[k].append(r)
            outs[k] = o
    res = {}
    for k in kinds:
        bpl = [bytes_fn(k.endswith("f32"), r) for r in runs[k]]
        res[k] = summarise(runs[k], bpl)
    res["outputs_identical"] = all(np.array_equal(u, v) for u, v in zip(outs[kinds[0]], outs[kinds[1]]))
    a, b = (min(res[k]["kernel_ms_per_launch"]["all"]) for k in kinds)
    res["kernel_ms_ratio_f32_over_f64"] = a / b
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=100000)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--max-iterations", type=int, default=100)
    ap.add_argument("--compare-tree", default=None, help="a built checkout to compare bench.py --config c3 against")
    ap.add_argument("--compare-label", default="other")
    ap.add_argument("--bench-rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import libdogleg_b200 as dlb
    from support import f32jac as HF
    from support import harness as H
    L = dlb.load()
    if L.dogleg_gpu_device_count() <= 0:
        raise SystemExit("no CUDA device: this measurement needs the GPU")
    doc = {"gpu": gpu_identity(), "hbm_peak_used_GBs": HBM_DATASHEET_GBS,
           "hbm_peak_source": "NVIDIA HGX B200 data sheet, per GPU (not a measured peak)",
           "callback": CALLBACK_NOTE,
           "double_form": "dogleg_gpu_optimize_dense_batched2 / _ragged with the widened twin callback",
           "rounds": args.rounds}
    B = args.batch

    # ---- (a), (b) C3's shape ----
    M = 256
    dev, p0 = HF.create(np.full(B, M, dtype=np.uint32), N, 3000)
    kinds = ("uniform_f32", "uniform_twin")
    per_launch = lambda f32, r: r["active_problem_launches"] / r["launches"] * per_problem_bytes(f32, M)  # noqa: E731
    doc["a_c3_full_solve"] = compare(HF, L, H, dev, p0, kinds, None, args.max_iterations, args.rounds, per_launch)
    doc["b_c3_first_launch"] = compare(HF, L, H, dev, p0, kinds, None, 0, args.rounds, per_launch)
    HF.free(dev)
    L.dogleg_gpu_release_batched_cache()

    # ---- (c) the skewed ragged batch ----
    counts = skewed_counts(B)
    dev, p0 = HF.create(counts, N, 5000)
    rows = float(counts.astype(np.int64).sum())
    kinds = ("ragged_f32", "ragged_twin")
    first = lambda f32, r: per_problem_bytes(f32, rows)  # noqa: E731  every problem active
    doc["c_skewed_ragged"] = {
        "counts": {"mean": float(counts.mean()), "min": int(counts.min()), "max": int(counts.max()), "rows": int(rows)},
        "first_launch": compare(HF, L, H, dev, p0, kinds, counts, 0, args.rounds, first),
        "full_solve": {k: v for k, v in compare(HF, L, H, dev, p0, kinds, counts, args.max_iterations, args.rounds,
                                                 lambda f32, r: float("nan")).items()}}
    for k in kinds:
        doc["c_skewed_ragged"]["full_solve"][k].pop("share_of_7p7TBs")
        doc["c_skewed_ragged"]["full_solve"][k].pop("algorithmic_bytes_per_launch")
    HF.free(dev)
    L.dogleg_gpu_release_batched_cache()

    # ---- (d) bench.py --config c3 against another tree ----
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
        ms = {k: [round(x["avg_launch_ms"], 4) for x in v] for k, v in bench.items()}
        doc["d_bench_c3_against_other_tree"] = {
            "other_tree": args.compare_label, "outputs_identical_every_round": identical,
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
