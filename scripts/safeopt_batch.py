#!/usr/bin/env python
"""Batch SafeOpt acquisition at C4 (d=4, 32^4 grid, n=512, G=4) on one GPU.

  The default C4 step (fantasy expander, tf32 with the FP64 refinement) runs once; then batches with q in {1, 4, 16, 64}
  are ALTERNATED, --reps repetitions each, on that step.  Batch time = host clock around sbo_safeopt_batch, which ends in a
  device synchronise (the picks are copied to the host).  Per q: median and range, kernel launches (sbo_kernel_launches),
  |C| = |M u E| and the work per pick computed from shapes: |C| n kernel evaluations and |C| (n (3d + 6) + q) flops (the
  downdate's c(p, x_b): per training point d differences, squares and scaled sums plus the kernel and its product with u_b;
  the correction over the earlier picks).  For comparison, one posterior pass over the grid (sbo_posterior, what a pick
  costs when it is made by appending a sample and rerunning the step) is timed the same way in the same process.  The GPU
  name and power limit are read in the same run.  One JSON line on stdout and in OUT/r04_safeopt_batch_c4_1gpu.json.
      python scripts/safeopt_batch.py --out DIR [--reps 5]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import sbo_b200  # noqa: E402
from sbo_b200 import _capi as capi, workloads  # noqa: E402

QS = (1, 4, 16, 64)


def gpu_info():
    r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="directory for the JSON line")
    ap.add_argument("--reps", type=int, default=5, help="alternated timed batches per q")
    a = ap.parse_args()
    ds, lo, hi, pts, beta = workloads.c4()
    n, d = ds["X_norm"].shape
    eng = sbo_b200.GridEngine(0)
    eng.set_grid(lo, hi, pts)
    t0 = time.perf_counter()
    st = eng.safeopt_step(ds, beta, mode="fantasy", precision="tf32", unsafe_rule=capi.UNSAFE_ANY)
    step_ms = (time.perf_counter() - t0) * 1e3
    ncand = eng.batch_prepare(1)               # |C| of the step (the staged prepare touches no step state)
    times = {q: [] for q in QS}
    launches, picks = {}, {}
    for q in QS:                               # warm-up of every shape
        eng.safeopt_batch(q)
    for _ in range(a.reps):
        for q in QS:
            eng.kernel_launches(reset=True)
            t = time.perf_counter()
            p = eng.safeopt_batch(q)
            times[q].append((time.perf_counter() - t) * 1e3)
            launches[q] = eng.kernel_launches()
            picks[q] = [x["idx"] for x in p]
    # one posterior pass over the grid, timed after the batches (it invalidates the step's sets)
    post = []
    for _ in range(a.reps + 1):
        t = time.perf_counter()
        eng.posterior(with_grad=False, keep_v=0, fetch=False)
        post.append((time.perf_counter() - t) * 1e3)
    post = post[1:]
    rows = {}
    for q in QS:
        rows[str(q)] = {"ms_median": statistics.median(times[q]), "ms_min": min(times[q]), "ms_max": max(times[q]),
                        "ms_per_pick": statistics.median(times[q]) / q, "launches": launches[q],
                        "kernel_evals_per_pick": ncand * n, "flops_per_pick": ncand * (n * (3 * d + 6) + q),
                        "picks": picks[q][:16]}
    out = {"workload": "c4", "gpu": gpu_info(), "reps": a.reps, "n": n, "d": d, "N": int(eng.N), "candidates": ncand,
           "n_safe": st["n_safe"], "n_min": st["n_min"], "expander_hits": st["expander"]["n_hit"], "x_new_idx": st["x_new_idx"],
           "step_ms_first_call": step_ms, "posterior_ms_median": statistics.median(post), "posterior_ms_min": min(post),
           "batch": rows}
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "r04_safeopt_batch_c4_1gpu.json"), "w") as f:
            f.write(line + "\n")
    eng.close()


if __name__ == "__main__":
    main()
