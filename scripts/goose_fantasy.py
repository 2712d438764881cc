#!/usr/bin/env python
"""Fantasy-mode GoOSE step (target set from the fantasy pair test, csrc/pairs.cu) on one GPU or sharded.

  one GPU, C4 (default): for tf32 (default refinement), tf32x3 and fp64 the GoOSE fantasy step is ALTERNATED with the
  SafeOpt fantasy step on the same model in this process, after warm-up; step time = host clock around a device-synchronised
  step.  Reports phase_ms (4 GEMM, 6 pair preparation, 7 FP64 refinement), launches, pair statistics, refine_stats, |T|, the
  target and x_new, and checks that the tf32 target set equals the fp64 one.  One JSON line on stdout and in
  OUT/goose_fantasy_<workload>_1gpu.json.
      python scripts/goose_fantasy.py --out DIR [--workload c4] [--reps 5]
  one GPU, one step in the format of the sharded run (the reference of a multi-GPU comparison):
      python scripts/goose_fantasy.py --workload c4s --sharded-reference [--refine 2]
  W GPUs, the sharded step (library communicator or the torch.distributed orchestrator):
      python -m torch.distributed.run --nproc-per-node 2 scripts/goose_fantasy.py --workload c4s --orchestrator library --refine 2
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
ap.add_argument("--workload", default="c4", choices=["c4", "c4s"])
ap.add_argument("--out", default=None, help="directory for the JSON line of the one-GPU measurement")
ap.add_argument("--reps", type=int, default=5, help="alternated timed steps per precision")
ap.add_argument("--precision", default="tf32", choices=["tf32", "tf32x3", "fp64"], help="sharded / reference runs")
ap.add_argument("--refine", type=int, default=2, choices=[2, 3], help="fantasy_refine of sharded / reference runs")
ap.add_argument("--orchestrator", default="library", choices=["library", "torch"])
ap.add_argument("--sharded-reference", action="store_true")
a = ap.parse_args()

distributed = "WORLD_SIZE" in os.environ               # started by torch.distributed.run (also with one process)
nproc = int(os.environ.get("WORLD_SIZE", "1"))
rank = int(os.environ.get("RANK", "0"))
local = int(os.environ.get("LOCAL_RANK", "0"))
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
if distributed:
    dist.init_process_group("nccl", device_id=dev)
ds, lo, hi, pts, beta = workloads.c4() if a.workload == "c4" else workloads.c4(pts_per_dim=16, n=128)
stream = torch.cuda.Stream(device=dev)
eng = sbo_b200.GridEngine(local, stream=stream.cuda_stream)
eng.set_grid(lo, hi, pts)
eng.set_model(ds)
rule = capi.UNSAFE_ALL


def summary(st):
    tg = st["target"]
    out = {k: int(st[k]) for k in ("n_safe", "n_unsafe", "target_idx", "x_new_idx", "explore_idx")}
    out.update({k: int(tg[k]) for k in ("n_hit", "n_x", "n_z", "pairs_evaluated", "n_ambiguous", "n_refined_safe", "n_undecided",
                                        "undecided_best_idx")})
    out["target_lcb"] = float(st["target_lcb"])
    return out


if distributed or a.sharded_reference:
    eng.set_option("fantasy_refine", a.refine)
    with torch.cuda.stream(stream):
        if distributed:
            eng.set_shard_cyclic(rank, nproc, 256)
            eng.set_model(ds)
            if a.orchestrator == "library":
                sharded.init_comm(eng, dev)
            st = sharded.goose_step(eng, ds, beta, unsafe_rule=rule, device=dev, mode="fantasy", precision=a.precision)
        else:
            st = eng.goose_step(ds, beta, rule, mode="fantasy", precision=a.precision)
    torch.cuda.synchronize()
    tg = st["target"]
    out = {"workload": a.workload, "world": nproc, "orchestrator": a.orchestrator if distributed else "one GPU",
           "precision": a.precision, "fantasy_refine": a.refine, "n_safe": int(st["n_safe"]), "n_unsafe": int(st["n_unsafe"]),
           "n_hit": int(tg["n_hit"]), "n_undecided": int(tg.get("n_undecided", 0)), "target_idx": int(st["target_idx"]),
           "x_new_idx": int(st["x_new_idx"]), "explore_idx": int(st["explore_idx"])}
    if rank == 0:
        print(json.dumps(out))
    eng.close()
    if distributed:
        dist.destroy_process_group()
    sys.exit(0)

q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit,clocks.max.sm",
                    "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
res = {"workload": "C4: d=4, N=32^4=2^20 grid, n=512, G=4 (3 constraints)" if a.workload == "c4" else "c4s: 16^4 grid, n=128",
       "gpu": q, "timing": "host clock around a device-synchronised step; median and spread of --reps alternated steps",
       "reps": a.reps, "precisions": {}}


def timed(fn):
    torch.cuda.synchronize()
    eng.kernel_launches(reset=True)
    t0 = time.perf_counter()
    with torch.cuda.stream(stream):
        r = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3, r, eng.kernel_launches(), eng.phase_ms(), eng.refine_stats()


masks = {}
for prec in ("tf32", "tf32x3", "fp64"):
    goose = lambda: eng.goose_step(ds, beta, rule, upload=False, mode="fantasy", precision=prec)      # noqa: E731
    safeopt = lambda: eng.safeopt_step(ds, beta, "fantasy", prec, rule, upload=False)                 # noqa: E731
    for _ in range(2):                                           # warm-up: modules, workspaces
        timed(goose)
        timed(safeopt)
    tg_ms, so_ms = [], []
    for _ in range(a.reps):
        ms, st, launches, ph, rs = timed(goose)
        tg_ms.append(ms)
        masks[prec] = eng.mask(capi.MASK_TARGET, 0)
        ms2, so, so_launches, so_ph, _ = timed(safeopt)
        so_ms.append(ms2)
    res["precisions"][prec] = {
        "goose_step_ms": {"median": statistics.median(tg_ms), "min": min(tg_ms), "max": max(tg_ms)},
        "safeopt_step_ms": {"median": statistics.median(so_ms), "min": min(so_ms), "max": max(so_ms)},
        "goose_phase_ms": {"gemm_4": ph["pairs"], "refine_7": ph["refine"], "pair_prep_6": ph["pair_prep"]},
        "safeopt_phase_ms": {"gemm_4": so_ph["pairs"], "refine_7": so_ph["refine"], "pair_prep_6": so_ph["pair_prep"]},
        "goose_launches": launches, "safeopt_launches": so_launches, "refine_stats": rs,
        "goose": summary(st), "safeopt_expander_n_hit": int(so["expander"]["n_hit"]), "safeopt_x_new_idx": int(so["x_new_idx"])}
res["checks"] = {"tf32_target_set_equals_fp64": bool(np.array_equal(masks["tf32"], masks["fp64"])),
                 "tf32x3_target_set_equals_fp64": bool(np.array_equal(masks["tf32x3"], masks["fp64"])),
                 "same_target_and_x_new": len({(p["goose"]["target_idx"], p["goose"]["x_new_idx"]) for p in res["precisions"].values()}) == 1}
line = json.dumps(res)
print(line)
if a.out:
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, f"goose_fantasy_{a.workload}_1gpu.json"), "w") as fh:
        fh.write(line + "\n")
eng.release(3)
eng.close()
assert all(res["checks"].values()), res["checks"]
