#!/usr/bin/env python
"""Incremental grid posterior (sbo_posterior_update) against the full posterior (sbo_posterior) at C4 on one GPU.

  The C4 recipe (workloads.c4: d=4, 32^4 grid, G=4) with n0 = 513 installed samples, so that up to 127 appends keep the padded
  factor at 640 rows; the appended samples are further draws of the same recipe, in the normalisation of the first 513.
  For m in {1, 4, 16, 64} appended samples and for keep_v = 0 (with_grad: the Lipschitz step's posterior) and keep_v = 2
  (TF32 V rows: the default fantasy step's), every repetition installs the n0-sample model, runs its posterior, appends m
  samples and then times, on that same appended model, sbo_posterior_update and then sbo_posterior (alternated, --reps
  each).  Times are host clocks around calls that end in a device synchronise.  Per case: median and range, kernel launches
  (sbo_kernel_launches), the work from shapes -- N n G kernel evaluations and N G (n (3d + 6) + 2 m n) flops of the update,
  n = n0 + m -- the posterior's own phases (phase_ms crosscov = K1a, solve) and the update's phase 8, and the check that the
  mean is bitwise equal and var within 1e-12 sf2 Y_std^2.  Then the whole Lipschitz SafeOpt step and the default fantasy step
  (tf32) after one append, with the update and with the full posterior (alternated), and the check that their expander sets
  and x_new agree.  The GPU name, power limit and max SM clock are read in the same run.  One JSON line on stdout and in
  OUT/r06_posterior_update_c4_1gpu.json.
      python scripts/posterior_update.py --out DIR [--reps 6]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import sbo_b200  # noqa: E402
from sbo_b200 import _capi as capi, workloads  # noqa: E402

N0 = 513
MS = (1, 4, 16, 64)
KEEP = {0: "keep_v0_with_grad", 2: "keep_v2_tf32"}


def gpu_info():
    r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip()


def timed(f):
    t = time.perf_counter()
    r = f()
    return (time.perf_counter() - t) * 1e3, r


def stats(v):
    return {"ms_median": statistics.median(v), "ms_min": min(v), "ms_max": max(v)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="directory for the JSON line")
    ap.add_argument("--reps", type=int, default=6, help="alternated calls per case; the first fetches and is checked, not timed")
    a = ap.parse_args()
    ds1, lo, hi, pts, beta = workloads.c4(n=N0 + max(MS))
    ds0 = dict(ds1, X_norm=ds1["X_norm"][:N0], Y_norm=ds1["Y_norm"][:N0])
    d, G = ds1["X_norm"].shape[1], ds1["Y_norm"].shape[1]
    sf2y2 = np.exp(2.0 * ds1["hypopt"][d]) * ds1["Y_std"] ** 2
    eng = sbo_b200.GridEngine(0)
    eng.set_grid(lo, hi, pts)
    N = int(eng.N)

    def install(m, with_grad, kv):
        eng.set_model(ds0)
        eng.posterior(with_grad=with_grad, keep_v=kv, fetch=False)
        for r in range(N0, N0 + m):
            eng.append_sample(ds1["X_norm"][r], ds1["Y_norm"][r])

    cases, checks = {}, {"mean_bitwise": True, "var_max_rel": 0.0}
    for m in MS:                                      # warm-up of every shape
        for kv in KEEP:
            install(m, kv == 0, kv)
            eng.posterior_update(fetch=False)
    for m in MS:
        n = N0 + m
        for kv, name in KEEP.items():
            tu, tf, lu, lf, ph_u, ph_f = [], [], [], [], [], []
            for rep in range(a.reps):
                install(m, kv == 0, kv)
                eng.kernel_launches(reset=True)
                t, (mv_u, info) = timed(lambda: eng.posterior_update(fetch=rep == 0))
                assert info["rows"] == m and not info["recomputed"], info
                tu.append(t)
                lu.append(eng.kernel_launches(reset=True))
                ph_u.append(eng.phase_ms()["posterior_update"])
                t, mv_f = timed(lambda: eng.posterior(with_grad=kv == 0, keep_v=kv, fetch=rep == 0))
                tf.append(t)
                lf.append(eng.kernel_launches(reset=True))
                ph = eng.phase_ms()
                ph_f.append((ph["crosscov"], ph["solve"]))
                if rep == 0:                          # the fetched runs are checked, not timed against the others
                    tu.pop(); tf.pop()
                    checks["mean_bitwise"] &= bool(np.array_equal(mv_u[0], mv_f[0]))
                    checks["var_max_rel"] = max(checks["var_max_rel"], float(np.max(np.abs(mv_u[1] - mv_f[1]) / sf2y2)))
            cases[f"m{m}_{name}"] = {
                "m": m, "n": n, "keep_v": kv, "with_grad": kv == 0,
                "update": dict(stats(tu), launches=lu[-1], phase8_ms_median=statistics.median(ph_u[1:])),
                "posterior": dict(stats(tf), launches=lf[-1], crosscov_k1a_ms_median=statistics.median(p[0] for p in ph_f[1:]),
                                  solve_ms_median=statistics.median(p[1] for p in ph_f[1:])),
                "speedup_median": statistics.median(tf) / statistics.median(tu),
                "kernel_evals": N * n * G, "update_flops": N * G * (n * (3 * d + 6) + 2 * m * n)}

    # whole steps after one append: Lipschitz SafeOpt step (with_grad) and the default fantasy step (tf32)
    def step(mode, use_update):
        fantasy = mode == "fantasy"
        prec, kv = capi.PRECISIONS["tf32"] if fantasy else (capi.PREC_FP64, 0)
        if use_update:
            eng.posterior_update(fetch=False)
        else:
            eng.posterior(with_grad=not fantasy, keep_v=kv, fetch=False)
        s = eng.sets(beta, capi.UNSAFE_ANY)
        if fantasy:
            ex = eng.expander(beta, None, capi.MODE_FANTASY, prec)
        else:
            L = np.full(G, eng.lipschitz()[G - 1])
            ex = eng.expander(beta, L, capi.MODE_LIPSCHITZ, prec)
        std_min = np.sqrt(s["minimizer_var"]) if s["minimizer_idx"] >= 0 else 0.0
        std_exp = np.sqrt(ex["best_value"]) if ex["best_idx"] >= 0 else 0.0
        x_new = s["minimizer_idx"] if std_min > std_exp else ex["best_idx"]
        masks = [eng.mask(capi.MASK_EXPANDER, c) for c in range(1 if fantasy else G - 1)]
        return x_new, ex["n_hit"], masks

    steps = {}
    for mode in ("lipschitz", "fantasy"):
        kv = 2 if mode == "fantasy" else 0
        for use_update in (True, False):              # warm-up
            install(1, kv == 0, kv)
            step(mode, use_update)
        tu, tf, same = [], [], True
        for _ in range(a.reps):
            install(1, kv == 0, kv)
            t, ru = timed(lambda: step(mode, True))
            tu.append(t)
            t, rf = timed(lambda: step(mode, False))
            tf.append(t)
            same &= ru[0] == rf[0] and ru[1] == rf[1] and all(np.array_equal(x, y) for x, y in zip(ru[2], rf[2]))
        steps[mode] = {"with_update": stats(tu), "with_posterior": stats(tf), "x_new_idx": int(ru[0]), "expander_hits": int(ru[1]),
                       "x_new_and_expander_equal": bool(same)}
    out = {"workload": "c4 recipe, n0 = 513", "gpu": gpu_info(), "reps_timed": a.reps - 1, "N": N, "d": d, "G": G, "n0": N0,
           "checks": checks, "cases": cases, "steps_after_one_append": steps}
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "r06_posterior_update_c4_1gpu.json"), "w") as f:
            f.write(line + "\n")
    eng.close()


if __name__ == "__main__":
    main()
