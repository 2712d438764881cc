#!/usr/bin/env python
"""Matern covariance functions at C4 (d=4, 32^4 grid, n=512, G=4) on one GPU.

  After warm-up, the C4 SafeOpt fantasy step in the default precision (tf32, FP64 refinement) is ALTERNATED for the SE,
  Matern 3/2 and Matern 5/2 kernels on the same data, grid and hyper-parameters; step time = host clock around a
  device-synchronised step.  Reports per kernel the median and range of the step, phase_ms (crosscov, solve, GEMM, pair
  preparation, refinement), launches, pairs_evaluated, n_ambiguous, refine_stats, n_hit and x_new; the Matern 5/2 GoOSE
  fantasy step; and checks that the tf32 and fp64 Matern expander sets are equal.  One JSON line on stdout and in
  OUT/matern_c4_1gpu.json, with the GPU name and power limit read in the same run.
      python scripts/matern_c4.py --out DIR [--reps 5]
  Two or more GPUs (test of the sharded step): the library-orchestrated Matern 5/2 fantasy SafeOpt and GoOSE steps on the 16^4
  grid against the one-GPU steps of rank 0; prints {"agree": ...}.
      python -m torch.distributed.run --nproc-per-node 2 scripts/matern_c4.py --sharded-check
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
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402
import sbo_b200  # noqa: E402
from sbo_b200 import _capi as capi, sharded, workloads  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--out", default=None, help="directory for the JSON line")
ap.add_argument("--reps", type=int, default=5, help="alternated timed steps per kernel")
ap.add_argument("--sharded-check", action="store_true")
a = ap.parse_args()
rule = capi.UNSAFE_ALL
KERNELS = ("RBF", "Matern32", "Matern52")

if a.sharded_check:
    nproc, rank, local = int(os.environ["WORLD_SIZE"]), int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    ds, lo, hi, pts, beta = workloads.c4(pts_per_dim=16, n=128)
    eng = sbo_b200.GridEngine(local)
    eng.set_grid(lo, hi, pts)
    eng.set_shard_cyclic(rank, nproc, 256)
    sharded.init_comm(eng, dev)
    keys = ("x_new_idx", "n_safe", "n_unsafe")
    sh = {m: sharded.safeopt_step(eng, ds, beta, mode=m, precision="tf32", kernel="Matern52") for m in ("lipschitz", "fantasy")}
    gs = sharded.goose_step(eng, ds, beta, mode="fantasy", precision="tf32", kernel="Matern52")
    if rank == 0:
        one = sbo_b200.GridEngine(local)
        one.set_grid(lo, hi, pts)
        ok = all(sh[m][k] == one.safeopt_step(ds, beta, mode=m, precision="tf32", kernel="Matern52")[k]
                 for m in sh for k in keys)
        g1 = one.goose_step(ds, beta, mode="fantasy", precision="tf32", kernel="Matern52")
        ok = ok and (gs["target_idx"], gs["x_new_idx"]) == (g1["target_idx"], g1["x_new_idx"])
        print(json.dumps({"world": nproc, "agree": bool(ok)}))
        one.close()
    eng.close()
    dist.destroy_process_group()
    sys.exit(0)

torch.cuda.set_device(0)
q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                   capture_output=True, text=True).stdout.strip()
ds, lo, hi, pts, beta = workloads.c4()
eng = sbo_b200.GridEngine(0)
eng.set_grid(lo, hi, pts)


def timed(fn):
    torch.cuda.synchronize()
    eng.kernel_launches(reset=True)
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3, r, eng.kernel_launches(), eng.phase_ms(), eng.refine_stats()


step = {k: (lambda k=k: eng.safeopt_step(ds, beta, mode="fantasy", precision="tf32", unsafe_rule=rule, kernel=k)) for k in KERNELS}
for _ in range(2):                                               # warm-up: modules, workspaces
    for k in KERNELS:
        timed(step[k])
ms = {k: [] for k in KERNELS}
last = {}
for _ in range(a.reps):
    for k in KERNELS:
        t, st, launches, ph, rs = timed(step[k])
        ms[k].append(t)
        last[k] = (st, launches, ph, rs)
res = {"workload": "C4: d=4, N=32^4=2^20 grid, n=512, G=4 (3 constraints), SafeOpt fantasy step, tf32 + FP64 refinement",
       "gpu": q, "timing": "host clock around a device-synchronised step; median and range of --reps steps, kernels alternated",
       "reps": a.reps, "kernels": {}}
for k in KERNELS:
    st, launches, ph, rs = last[k]
    ex = st["expander"]
    res["kernels"][k] = {
        "step_ms": {"median": statistics.median(ms[k]), "min": min(ms[k]), "max": max(ms[k])},
        "phase_ms": {"crosscov": ph["crosscov"], "solve": ph["solve"], "gemm": ph["pairs"], "pair_prep": ph["pair_prep"],
                     "refine": ph["refine"]},
        "launches": launches, "pairs_evaluated": int(ex["pairs_evaluated"]), "n_ambiguous": int(ex["n_ambiguous"]),
        "n_refined_safe": int(ex["n_refined_safe"]), "refine_stats": rs, "n_hit": int(ex["n_hit"]),
        "n_safe": int(st["n_safe"]), "n_unsafe": int(st["n_unsafe"]), "x_new_idx": int(st["x_new_idx"])}
# GoOSE fantasy step, Matern 5/2
gms = []
for _ in range(a.reps):
    t, g, launches, ph, rs = timed(lambda: eng.goose_step(ds, beta, rule, mode="fantasy", precision="tf32", kernel="Matern52"))
    gms.append(t)
tg = g["target"]
res["goose_matern52"] = {"step_ms": {"median": statistics.median(gms), "min": min(gms), "max": max(gms)},
                         "phase_ms": {"gemm": ph["pairs"], "pair_prep": ph["pair_prep"], "refine": ph["refine"]},
                         "launches": launches, "n_hit": int(tg["n_hit"]), "n_ambiguous": int(tg["n_ambiguous"]),
                         "n_refined_safe": int(tg["n_refined_safe"]), "refine_stats": rs,
                         "target_idx": int(g["target_idx"]), "x_new_idx": int(g["x_new_idx"])}
# the tf32 (refined) and fp64 Matern expander sets
checks = {}
for k in ("Matern32", "Matern52"):
    sets = {}
    for prec in ("tf32", "fp64"):
        st = eng.safeopt_step(ds, beta, mode="fantasy", precision=prec, unsafe_rule=rule, kernel=k)
        sets[prec] = (eng.mask(capi.MASK_EXPANDER, 0), int(st["x_new_idx"]))
    checks[f"{k}_tf32_expander_set_equals_fp64"] = bool(np.array_equal(sets["tf32"][0], sets["fp64"][0]))
    checks[f"{k}_same_x_new"] = sets["tf32"][1] == sets["fp64"][1]
res["checks"] = checks
line = json.dumps(res)
print(line)
if a.out:
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "matern_c4_1gpu.json"), "w") as fh:
        fh.write(line + "\n")
eng.release(3)
eng.close()
assert all(checks.values()), checks
