#!/usr/bin/env python
"""Batch GoOSE acquisition at C4 (d=4, 32^4 grid, n=512, G=4) on one GPU.

  The C4 GoOSE step (fantasy target, tf32 with the FP64 refinement) runs once; then batches with q in {1, 4, 16, 64} are
  ALTERNATED, --reps repetitions each, on that step.  Batch time = host clock around sbo_goose_batch, which ends in a device
  synchronise (the picks are copied to the host).  Per q: median and range, kernel launches (sbo_kernel_launches), the
  explore / safe mix and the number of distinct targets served.  |C| = |S u T| and the work per pick from shapes: |C| n
  kernel evaluations.  In the same process, the SafeOpt batch (sbo_safeopt_batch) on the default SafeOpt step of the same
  model, timed the same way, and one posterior pass over the grid (sbo_posterior, what a pick costs when it is made by
  appending a sample and rerunning the step).  The GPU name and power limit are read in the same run.  One JSON line on
  stdout and in OUT/r05_goose_batch_c4_1gpu.json.
      python scripts/goose_batch.py --out DIR [--reps 5]
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


def timed_batches(eng, fn, reps):
    """Warm every q, then `reps` alternated rounds over QS: {q: (times ms, launches, picks)}."""
    for q in QS:
        fn(q)
    times = {q: [] for q in QS}
    launches, picks = {}, {}
    for _ in range(reps):
        for q in QS:
            eng.kernel_launches(reset=True)
            t = time.perf_counter()
            p = fn(q)
            times[q].append((time.perf_counter() - t) * 1e3)
            launches[q] = eng.kernel_launches()
            picks[q] = p
    return times, launches, picks


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="directory for the JSON line")
    ap.add_argument("--reps", type=int, default=5, help="alternated timed batches per q")
    a = ap.parse_args()
    gpu = gpu_info()
    ds, lo, hi, pts, beta = workloads.c4()
    n, d = ds["X_norm"].shape
    eng = sbo_b200.GridEngine(0)
    eng.set_grid(lo, hi, pts)
    t0 = time.perf_counter()
    st = eng.goose_step(ds, beta, mode="fantasy", precision="tf32", unsafe_rule=capi.UNSAFE_ANY)
    step_ms = (time.perf_counter() - t0) * 1e3
    ncand = eng.goose_batch_prepare(1)         # |C| of the step (the staged prepare touches no step state)
    times, launches, picks = timed_batches(eng, eng.goose_batch, a.reps)
    rows = {}
    for q in QS:
        p = picks[q]
        rows[str(q)] = {"ms_median": statistics.median(times[q]), "ms_min": min(times[q]), "ms_max": max(times[q]),
                        "ms_per_pick": statistics.median(times[q]) / q, "launches": launches[q], "n_picked": len(p),
                        "explore": sum(x["explore"] for x in p), "safe": sum(1 - x["explore"] for x in p),
                        "distinct_targets": len({x["target_idx"] for x in p if x["explore"]}),
                        "distinct_picks": len({x["idx"] for x in p}), "kernel_evals_per_pick": ncand * n,
                        "picks": [x["idx"] for x in p][:16]}
    # the SafeOpt batch on the default SafeOpt step of the same model, timed the same way
    so = eng.safeopt_step(ds, beta, mode="fantasy", precision="tf32", unsafe_rule=capi.UNSAFE_ANY)
    so_cand = eng.batch_prepare(1)
    so_times, so_launches, _ = timed_batches(eng, eng.safeopt_batch, a.reps)
    so_rows = {str(q): {"ms_median": statistics.median(so_times[q]), "ms_min": min(so_times[q]), "ms_max": max(so_times[q]),
                        "ms_per_pick": statistics.median(so_times[q]) / q, "launches": so_launches[q]} for q in QS}
    # one posterior pass over the grid, timed after the batches (it invalidates the step's sets)
    post = []
    for _ in range(a.reps + 1):
        t = time.perf_counter()
        eng.posterior(with_grad=False, keep_v=0, fetch=False)
        post.append((time.perf_counter() - t) * 1e3)
    post = post[1:]
    out = {"workload": "c4", "gpu": gpu, "gpu_after": gpu_info(), "reps": a.reps, "n": n, "d": d, "N": int(eng.N),
           "candidates": ncand, "n_safe": st["n_safe"], "target_hits": st["target"]["n_hit"], "x_new_idx": st["x_new_idx"],
           "explore_idx": st["explore_idx"], "step_ms_first_call": step_ms, "goose_batch": rows,
           "safeopt_candidates": so_cand, "safeopt_x_new_idx": so["x_new_idx"], "safeopt_batch": so_rows,
           "posterior_ms_median": statistics.median(post), "posterior_ms_min": min(post)}
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "r05_goose_batch_c4_1gpu.json"), "w") as f:
            f.write(line + "\n")
    eng.close()


if __name__ == "__main__":
    main()
