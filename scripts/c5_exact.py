#!/usr/bin/env python
"""C5 (d=6, N=16^6=2^24, n=2048, G=4) fantasy step in bounds mode (fantasy_refine = 3) and in exact mode (fantasy_refine = 2,
the FP64 refinement cut into cells when its rows do not fit), with the bracket checks between them.  One JSON line on stdout
and the same line in OUT/c5_exact_<topology>.json.

  one GPU as rank r of W (default 0 of 8, like c5_shard_probe.py: the rank's shard, its local candidates x its local unsafe
  points), in one process:  1. bounds mode   2. exact, automatic budget   3. exact, --refine-mb budget
      python scripts/c5_exact.py --out DIR [--rank 0 --world 8 --refine-mb 4096]
  W GPUs, the whole sharded step with the library communicator:  1. bounds mode   2. exact, automatic budget
      python -m torch.distributed.run --nproc-per-node 8 scripts/c5_exact.py --out DIR

Checks: the exact n_hit lies in [certified, certified + undecided]; on one GPU also that runs 2 and 3 give identical counts
and x_new and that every certified candidate has an exact count > 0."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402
import sbo_b200  # noqa: E402
from sbo_b200 import _capi as capi, sharded, workloads  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--out", required=True, help="directory for c5_exact_<topology>.json")
ap.add_argument("--world", type=int, default=8, help="one-GPU mode: the shard is rank --rank of --world")
ap.add_argument("--rank", type=int, default=0)
ap.add_argument("--refine-mb", type=int, default=4096, help="one-GPU mode: the forced budget of run 3")
a = ap.parse_args()

nproc = int(os.environ.get("WORLD_SIZE", "1"))
rank = int(os.environ.get("RANK", "0"))
local = int(os.environ.get("LOCAL_RANK", "0"))
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
if nproc > 1:
    dist.init_process_group("nccl", device_id=dev)
ds, lo, hi, pts, beta = workloads.c5()
stream = torch.cuda.Stream(device=dev)
eng = sbo_b200.GridEngine(local, stream=stream.cuda_stream)
eng.set_grid(lo, hi, pts)
if nproc > 1:
    eng.set_shard_cyclic(rank, nproc, 256)
    with torch.cuda.stream(stream):
        sharded.init_comm(eng, dev)
    topo = f"{nproc}gpu"
else:
    eng.set_shard_cyclic(a.rank, a.world, 256)
    topo = f"1gpu_rank{a.rank}of{a.world}"
q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit,clocks.max.sm",
                    "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
out = {"workload": "C5: d=6, N=16^6=2^24 grid, n=2048, G=4 (3 constraints)", "precision": "tf32", "topology": topo,
       "gpu": q, "device_mem_total_gb": torch.cuda.mem_get_info(dev)[1] / 2 ** 30, "runs": {}}


def step(refine, mb):
    """One fantasy SafeOpt step; returns (result, counts or None, device ms)."""
    eng.set_option("fantasy_refine", refine)
    eng.set_option("fantasy_refine_mb", mb)
    eng.mem_peak(reset=True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(stream):
        e0.record(stream)
        if nproc > 1:
            r, counts = eng.safeopt_step_sharded(ds, beta, mode="fantasy", precision="tf32"), None
            ex = r["expander"]
        else:                              # safeopt_step's sequence, keeping the per-candidate counts
            prec, kv = capi.PRECISIONS["tf32"]
            eng.set_model(ds)
            eng.posterior(keep_v=kv, fetch=False)
            r = eng.sets(beta, capi.UNSAFE_ALL)
            ex = eng.expander(beta, None, capi.MODE_FANTASY, prec, want_counts=True)
            counts = ex.pop("counts")
            mstd = float(np.sqrt(r["minimizer_var"])) if r["minimizer_idx"] >= 0 else 0.0
            estd = float(np.sqrt(ex["best_value"])) if ex["best_idx"] >= 0 else 0.0
            r["x_new_idx"] = r["minimizer_idx"] if mstd > estd else ex["best_idx"]
            r["expander"] = ex
        e1.record(stream)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if nproc > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t[0])
    rep = {"fantasy_refine": refine, "fantasy_refine_mb": mb, "ms_per_step": ms, "phase_ms": eng.phase_ms(),
           "refine_stats": eng.refine_stats(), "mem_peak_gb": eng.mem_peak() / 2 ** 30,
           "n_safe": int(r["n_safe"]), "n_unsafe": int(r["n_unsafe"]), "n_hit": int(ex["n_hit"]), "x_new_idx": int(r["x_new_idx"]),
           "n_ambiguous": int(ex["n_ambiguous"]), "n_refined_safe": int(ex["n_refined_safe"])}
    if refine == 3:
        rep.update({"certified": int(ex["n_hit"]), "undecided": int(ex["n_undecided"])})
    return rep, counts


eng.set_option("fantasy_refine", 3)                        # warm-up: modules, workspaces
with torch.cuda.stream(stream):
    eng.safeopt_step_sharded(ds, beta, mode="fantasy", precision="tf32") if nproc > 1 else \
        eng.safeopt_step(ds, beta, mode="fantasy", precision="tf32")
torch.cuda.synchronize()
plan = [("bounds", 3, 0), ("exact_auto", 2, 0)] + ([("exact_forced", 2, a.refine_mb)] if nproc == 1 else [])
counts = {}
for name, refine, mb in plan:
    out["runs"][name], counts[name] = step(refine, mb)
b, e = out["runs"]["bounds"], out["runs"]["exact_auto"]
checks = {"exact_n_hit_in_bracket": b["certified"] <= e["n_hit"] <= b["certified"] + b["undecided"]}
if nproc == 1:
    f = out["runs"]["exact_forced"]
    checks["forced_cells_gt_1"] = f["refine_stats"]["cells"] > 1
    checks["forced_counts_identical"] = bool(np.array_equal(counts["exact_auto"], counts["exact_forced"]))
    checks["forced_x_new_identical"] = f["x_new_idx"] == e["x_new_idx"] and f["n_hit"] == e["n_hit"]
    checks["certified_are_exact_members"] = bool(np.all(counts["exact_auto"][counts["bounds"] > 0] > 0))
out["checks"] = checks
if rank == 0:
    line = json.dumps(out)
    print(line)
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, f"c5_exact_{topo}.json"), "w") as fh:
        fh.write(line + "\n")
eng.close()
if nproc > 1:
    dist.destroy_process_group()
assert all(checks.values()), checks
