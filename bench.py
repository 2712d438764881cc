#!/usr/bin/env python
"""bench.py -- SafeOpt/GoOSE grid step on N B200s: expander pair-evals/s (+ step time).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload c4|c5|c4s] [--mode fantasy|lipschitz] [--precision tf32|tf32x3|fp64]
                    [--dump-outputs DIR]

A "step" = model upload -> GP posterior over the grid for all G GPs -> safe/minimiser/unsafe sets ->
Lipschitz constants (Lipschitz mode) -> expander pair kernel -> arg-reductions -> x_new.  It EXCLUDES the
plant evaluation and the hyper-parameter fit, which stay on the host in the reference too.
Workload at N=1: BASELINE.json configs[3] "synthetic SafeOpt expander step: 2^20-point d=4 grid, n=512
observations, 3 constraint GPs" (C4); the grid is sharded over the ranks (strong scaling, fixed N).
`value` = pair-evals of the whole job / device time of the step (CUDA events on the launch stream, every timed step
preceded by a barrier, max over ranks); `e2e` = the same through GridEngine.safeopt_step / sharded.safeopt_step with
HOST buffers (model H2D, result and safe-mask D2H inside the timed region, wall clock around a device sync).
Extra keys: `roofline` (the fantasy GEMM against the measured TF32 peak, DRAM traffic from the committed ncu capture),
`cpu_baseline` (N=1: the oracle on the host cores on a bounded sample), `lipschitz_mode` (step time of the
reference-exact SafeOpt and GoOSE steps on the same workload, any N), `reference_configs` (N=1: C1-C3, the
reference's own problems on its 400x400 grid), `phase_ms`, `clocks`, `gpu_launches`.
--impl reference times the NumPy oracle (the port of the reference's arithmetic; JAX is not installed)
on the host cores on a bounded sample of the same workload.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--workload", default="c4")
    ap.add_argument("--mode", default=os.environ.get("SBO_BENCH_MODE", "fantasy"))
    ap.add_argument("--precision", default=os.environ.get("SBO_BENCH_PRECISION", "tf32"),
                    help="fantasy GEMM operands: tf32 (default: single TF32 pass; every pair inside its error bound is re-evaluated in FP64, "
                         "so the counts are the FP64 counts), tf32x3 (split TF32, same refinement with a 100x narrower band), fp64 (DMMA)")
    ap.add_argument("--refine", type=int, default=2, help="FP64 refinement of the tensor-core modes: 2 (library default) tf32 and tf32x3, 1 tf32x3 only, 0 off, 3 bounds mode (classify only)")
    ap.add_argument("--e2e-steps", type=int, default=None, help="end-to-end repetitions (default max(2, steps); the first is dropped when > 1)")
    ap.add_argument("--orchestrator", default="library", choices=["library", "torch"],
                    help="multi-GPU: collectives inside libsbo_b200 (sbo_comm_init, default) or issued by sharded.py through torch.distributed")
    ap.add_argument("--c5", type=int, default=-1, help="1: add the C5 north-star step (2^24-point d=6 grid, n=2048) as an extra key; "
                    "default: on at --gpus 8 (the configuration BASELINE.json states the target on), off otherwise")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-peaks", action="store_true")
    ap.add_argument("--no-lipschitz-steps", action="store_true", help="skip the reference-exact SafeOpt/GoOSE step times (extra key)")
    ap.add_argument("--no-reference-configs", action="store_true", help="skip the C1-C3 step times (extra key)")
    ap.add_argument("--prune", type=int, default=1, help="exact key-ordered tile pruning of the fantasy expander (default 1 = the library default; 0 = every pair)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (rank 0; see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    return args


def workload(name):
    import sbo_b200  # noqa: F401
    from sbo_b200 import workloads
    if name == "c4":
        return workloads.c4(), "C4: synthetic SafeOpt expander step, d=4, N=32^4=2^20 grid, n=512, G=4 (3 constraints)"
    if name == "c5":
        return workloads.c5(), "C5: synthetic step, d=6, N=16^6=2^24 grid, n=2048, G=4 (3 constraints)"
    if name == "c4s":
        return workloads.c4(pts_per_dim=16, n=128), "C4-small: d=4, N=16^4, n=128, G=4 (debug size)"
    raise SystemExit(f"unknown workload {name}")


# --------------------------------------------------------------------------------------------
# clocks sampler (B200_PROFILING.md "clocks line")
# --------------------------------------------------------------------------------------------
class Clocks:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []                     # (arrival time, fields)
        self.proc = None
        self.t0 = None

    def start(self):
        """Launch the sampler (before the warm-up steps: nvidia-smi needs a few hundred ms to deliver its first row, more than a
        whole timed region at 8 GPUs)."""
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def mark(self):
        """Start of the timed region: only rows that arrive from here on are used (waits, bounded, for the sampler's first row)."""
        t = time.perf_counter()
        while self.proc is not None and not self.rows and time.perf_counter() - t < 2.0:
            time.sleep(0.01)
        self.t0 = time.perf_counter()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        t1 = time.perf_counter()
        time.sleep(0.12)                   # a row that was sampled inside the region may still be in the pipe
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        t0 = self.t0 if self.t0 is not None else 0.0
        inside = [r for t, r in self.rows if t0 <= t <= t1 + 0.06]
        window = "timed region"
        if not inside and self.rows:       # region shorter than the sampling period: the rows next to it (warm-up steps run right before)
            inside = [r for _, r in self.rows[-2:]]
            window = "nearest samples (timed region shorter than the sampling period)"
        sm, mx, reasons = [], [], set()
        for r in inside:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for nm, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "window": window}


# --------------------------------------------------------------------------------------------
# CPU arm: the oracle (NumPy port of the reference's arithmetic) on a bounded sample
# --------------------------------------------------------------------------------------------
# sample sizes: per --impl reference step (the driver runs 25 of them: a few seconds each) and for the one-off
# cpu_baseline of our arm (10-30 s of CPU work)
REF_STEP_SAMPLE = dict(n_points=16384, n_x=2048, n_z=16384)
CPU_BASELINE_SAMPLE = dict(n_points=65536, n_x=4096, n_z=40960)


def use_all_host_threads():
    """torchrun exports OMP_NUM_THREADS=1 to its workers; the CPU arm is meant to use every host core, so raise the
    BLAS / OpenMP thread counts back at run time.  Returns the number of threads in use."""
    n = os.cpu_count() or 1
    try:
        from threadpoolctl import threadpool_info, threadpool_limits
        threadpool_limits(limits=n)
        used = [i["num_threads"] for i in threadpool_info()]
        return max(used) if used else n
    except Exception:
        return int(os.environ.get("OMP_NUM_THREADS", n))


def full_pairs(args, ds, pts):
    """(N, |S|*|Z|*(G-1)) of the full workload.  |S|, |Z| are the GPU-computed set sizes recorded in BASELINE.md for
    the frozen workloads (identical to the oracle's on the same inputs, tests/test_gpu_parity.py)."""
    N = int(np.prod(pts))
    G = ds["Y_norm"].shape[1]
    known = {"c4": (116645, 757532), "c5": (1672419, 12956616)}
    if args.workload in known:
        ns, nz = known[args.workload]
        return N, ns * nz * (G - 1), "set sizes of the full workload (BASELINE.md)"
    return N, None, "set sizes estimated from the sample's safe/unsafe fractions"


def run_reference(args):
    """--impl reference: the reference's CPU arithmetic (oracle port; JAX is not installed, the reference itself cannot
    run) on the host cores.  Each step is a bounded sample of the workload; per-point and per-pair work are timed
    separately and each is extrapolated to the full step by its own ratio (oracle/cpu_arm.py)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import cpu_arm
    (ds, lo, hi, pts, beta), wl_name = workload(args.workload)
    G = ds["Y_norm"].shape[1]
    N, pairs_full, how = full_pairs(args, ds, pts)
    cores = use_all_host_threads()
    times, samples = [], []
    for it in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        s = cpu_arm.sample_step(ds, lo, hi, pts, beta, args.mode, seed=it, **REF_STEP_SAMPLE)
        dt = time.perf_counter() - t0
        if it >= args.warmup:
            times.append(dt); samples.append(s)
    if pairs_full is None:
        sf = float(np.mean([x["safe_frac"] for x in samples])); uf = float(np.mean([x["unsafe_frac"] for x in samples]))
        pairs_full = sf * N * uf * N * (G - 1)
    t_full = float(np.mean([cpu_arm.extrapolate(x, N, pairs_full) for x in samples]))
    s = samples[-1]
    value = pairs_full / t_full
    sample_desc = cpu_arm.describe(s, N, pairs_full, args.mode) + f"; per step, {len(samples)} timed steps with different seeds; {how}"
    line = {"impl": "reference", "metric": "expander_pair_evals_per_s", "value": value, "unit": "pair-evals/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": float(np.mean(times)) * 1e3,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": wl_name, "mode": args.mode,
                       "note": "NumPy/OpenBLAS restatement of the reference's arithmetic (oracle port), not JAX; ms_per_step is the "
                               "measured time of one bounded sample step, value = full-workload pairs / extrapolated full-step time"},
            "ms_per_step_extrapolated": t_full * 1e3,
            "pair_evals_per_s_pair_stage_only": float(np.mean([x["pairs"] / x["t_pairs"] for x in samples if x["t_pairs"] > 0] or [0.0])),
            "cpu_baseline": {"value": value, "unit": "pair-evals/s", "cores": cores, "kind": "port", "sample": sample_desc},
            "e2e": {"value": value, "unit": "pair-evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# --------------------------------------------------------------------------------------------
# BASELINE.json configs[0..2]: the reference's own problems on its 400x400 grid (step time part of the metric)
# --------------------------------------------------------------------------------------------
# B-DE context (BASELINE.md section 3): the reference-shaped step -- SciPy DE + NonlinearConstraint lambdas over a
# single-point inference (oracle/de_step.py restates models/SafeOpt.py:47-124, GoOSE.py:63-119) -- is timed in this
# run on the host next to the GPU step.  maxiter caps bound the time; a capped run is a lower bound of the reference's.
DE_MAXITER = {"C1 SafeOpt/Benoit n=14": 1000, "C2 GoOSE/Benoit n=14": 1000, "C3 SafeOpt/WOR n=35": 25}


def reference_configs(eng, torch, reps=5, with_de=True):
    """Step time (host wall clock around a device sync, model upload included) of one SafeOpt / GoOSE acquisition
    step in the reference-exact Lipschitz mode on the reference's 400x400 grid, for the model states the
    reference's own source produced (tests/golden/ref_*.npz)."""
    out = {}
    gdir = os.path.join(ROOT, "tests", "golden")
    cases = [("C1 SafeOpt/Benoit n=14", "ref_c1_benoit.npz", 14, "safeopt"),
             ("C2 GoOSE/Benoit n=14", "ref_c1_benoit.npz", 14, "goose"),
             ("C3 SafeOpt/WOR n=35", "ref_c3_wor.npz", 35, "safeopt")]
    for name, f, n, kind in cases:
        try:
            r = np.load(os.path.join(gdir, f))
            ds = {k: r[f"{k}_{n}"] for k in ("X_mean", "X_std", "Y_mean", "Y_std", "X_norm", "Y_norm", "hypopt")}
            beta = float(r["beta"])
            eng.set_grid(r["bound"][:, 0], r["bound"][:, 1], [400, 400])
            step = (lambda: eng.safeopt_step(ds, beta)) if kind == "safeopt" else (lambda: eng.goose_step(ds, beta))
            st = step()
            torch.cuda.synchronize()
            ts = []
            for _ in range(reps):
                t0 = time.perf_counter()
                st = step()
                torch.cuda.synchronize()
                ts.append(time.perf_counter() - t0)
            pr = st["expander"] if kind == "safeopt" else st["target"]
            out[name] = {"ms_per_step": float(np.median(ts)) * 1e3, "grid": "400x400", "mode": "lipschitz", "G": int(ds["Y_norm"].shape[1]),
                         "n_safe": int(st["n_safe"]), "n_unsafe": int(st["n_unsafe"]), "pairs": int(pr["pairs_algorithmic"]),
                         "pairs_evaluated": int(pr["pairs_evaluated"]), "x_new_idx": int(st["x_new_idx"])}
            if with_de:
                from oracle import de_step, gp_oracle as O
                dso = dict(ds)
                dso["invKopt"] = [np.linalg.inv(O.build_K(ds["X_norm"], ds["hypopt"][:, i])) for i in range(ds["Y_norm"].shape[1])]
                de = de_step.time_step(dso, r["bound"], beta, kind, seed=0, maxiter=DE_MAXITER[name])
                out[name]["reference_shaped_de_step"] = {
                    "seconds": de["seconds"], "single_point_inferences": de["n_inference"], "maxiter": de["maxiter"],
                    "capped_lower_bound": bool(de["capped"]),
                    "what": "SciPy DE + NonlinearConstraint over single-point NumPy inference, 1 host thread, timed in this run"}
        except Exception as e:  # pragma: no cover
            out[name] = {"error": str(e)}
    return out


# --------------------------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------------------------
# dram__bytes_read.sum + dram__bytes_write.sum of k_fantasy_tc per launch from the committed ncu capture
# (profiles/): filled in when a capture of the same configuration exists, else null
TRAFFIC_NCU = {
    # profiles/r02_ncu_fantasy_tc2_tf32r_summary.csv: tc::k_fantasy_tc2<1,8,refine> on C4, single TF32 pass over the tile pairs the
    # exact pruning keeps (one launch = the whole pair stage): 42.15 GB read + 0.04 GB written (3.2 % of the HBM bandwidth)
    ("c4", "tf32"): 42.146603e9 + 0.040392e9,
    # profiles/r02_ncu_fantasy_tc2_tf32x3_summary.csv (split operands, 2x the bytes per row): 227.7 GB read + 5.8 GB written
    ("c4", "tf32x3"): 227.733712e9 + 5.802020e9,
}


def measure_peaks(torch, dev):
    """Yard-sticks for the roofline denominators MEASURED_PEAKS.json lacks: cuBLAS FP64 and TF32 GEMM."""
    out = {}
    try:
        torch.backends.cuda.matmul.allow_tf32 = True
        for name, dt, n in (("fp64_tflops", torch.float64, 4096), ("tf32_tflops", torch.float32, 8192)):
            a = torch.randn(n, n, device=dev, dtype=dt); b = torch.randn(n, n, device=dev, dtype=dt)
            for _ in range(2):
                torch.matmul(a, b)
            best = 1e9
            for _ in range(5):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(); torch.matmul(a, b); e1.record(); torch.cuda.synchronize()
                best = min(best, e0.elapsed_time(e1))
            out[name] = 2.0 * n ** 3 / (best * 1e-3) / 1e12
            del a, b
    except Exception as e:  # pragma: no cover
        out["error"] = str(e)
    return out


def c5_key(args, eng, torch, dist, stream, rank, world, dev, barrier):
    """BASELINE.json configs[4] / the north-star target: one warm-up + one timed SafeOpt fantasy step on the 2^24-point
    d=6 grid with n=2048 observations, grid-sharded over the ranks.  Single-pass TF32 with the exact pruning: the
    split-TF32 operands (2 x 41 GB of gathered candidate rows) do not fit next to the z side at this size."""
    from sbo_b200 import workloads, sharded
    ds5, lo5, hi5, pts5, beta5 = workloads.c5()
    n5, d5 = ds5["X_norm"].shape
    out = {"workload": "C5: synthetic step, d=6, N=16^6=2^24 grid, n=2048, G=4 (3 constraints)", "precision": "tf32", "refine": "3 (bounds)", "n_gpus": world}
    try:
        eng.release(3)
        torch.cuda.empty_cache()
        # bounds mode at this size: the TF32 band holds ~3e8 pairs per rank here and their FP64 re-evaluation at n = 2048 would
        # gather ~30 TB of rows per rank, so the refining epilogue only CLASSIFIES -- the expander set is reported as the
        # candidates with a pair settled newly safe (certified members of the FP64 set) plus the count of undecided ones
        eng.set_option("fantasy_refine", 3 if (world == 1 or getattr(eng, "comm_ready", False)) else 0)
        if not (world == 1 or getattr(eng, "comm_ready", False)):
            out["refine"] = 0
        eng.set_grid(lo5, hi5, pts5)
        if world > 1:
            eng.set_shard_cyclic(rank, world, 256)
        free0, total = torch.cuda.mem_get_info(dev)
        # every rank must have the head-room (the step peaks at ~135 GB per GPU on 8): agree BEFORE any collective of the
        # step is entered, so that a rank that cannot run it does not leave the others waiting
        need = (135 << 30) * 8 // max(world, 8) if world >= 8 else (1 << 62)
        ok = torch.tensor([1 if free0 >= need else 0], dtype=torch.int32, device=dev)
        if world > 1:
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if int(ok[0]) == 0:
            out["skipped"] = f"needs {need >> 30} GB free per GPU on >= 8 GPUs (free here: {free0 >> 30} GB, {world} ranks)"
            return out

        def step5():
            with torch.cuda.stream(stream):
                if world == 1:
                    return eng.safeopt_step(ds5, beta5, mode="fantasy", precision="tf32")
                return sharded.safeopt_step(eng, ds5, beta5, mode="fantasy", precision="tf32")
        eng.mem_peak(reset=True)
        step5()
        torch.cuda.synchronize()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            e0.record(stream)
            r5 = step5()
            e1.record(stream)
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t[0])
        ph = eng.phase_ms()
        ex5 = r5["expander"]
        pairs5, ev5 = int(ex5["pairs_algorithmic"]), int(ex5["pairs_evaluated"])
        flops = ev5 / world * (2.0 * n5 + 3 * d5 + 20)
        mp = {}
        try:
            mp = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = mp.get("bf16_tflops_sustained", 1387.2) / 2.0
        ach = flops / (ph["pairs"] * 1e-3) / 1e12 if ph["pairs"] > 0 else None
        out.update({"ms_per_step": ms, "value": pairs5 / (ms * 1e-3), "unit": "pair-evals/s", "pairs": pairs5, "pairs_evaluated": ev5,
                    "n_safe": int(r5["n_safe"]), "n_unsafe": int(r5["n_unsafe"]), "n_min": int(r5["n_min"]), "n_hit": int(ex5["n_hit"]),
                    "x_new_idx": int(r5["x_new_idx"]), "phase_ms_rank0": ph,
                    "expander_bounds": {"certified_members": int(ex5["n_hit"]), "undecided_candidates": int(ex5.get("n_undecided", 0)),
                                        "pairs_inside_error_bound": int(ex5.get("n_ambiguous", 0)),
                                        "x_new_certified": bool(int(ex5.get("n_undecided", 0)) == 0 or
                                                                ex5.get("undecided_best_value", -np.inf) < max(ex5["best_value"], r5["minimizer_var"])),
                                        "note": "FP64 expander set = certified members + a subset of the undecided candidates"},
                    "roofline": {"bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak if ach else None,
                                 "kernel": "tc::k_fantasy_tc2 (tf32), per GPU, evaluated pairs only"},
                    "device_mem_high_water_gb": eng.mem_peak() / 2 ** 30,
                    "device_mem_total_gb": total / 2 ** 30, "steps": 1, "warmup": 1})
        # parity at full size: this rank's posterior on a random sample of its shard against the FP64 oracle
        if rank == 0:
            from oracle import gp_oracle as O
            m, v = eng.posterior(keep_v=0)
            rng = np.random.default_rng(0)
            cnt = eng.count
            sel = np.sort(rng.choice(cnt, size=128, replace=False))
            sb = sel // 256
            gidx = ((sb * world + (rank + sb + sb // world + sb // (world * world)) % world) * 256 + sel % 256) if world > 1 else sel
            axes = O.grid_axes(lo5, hi5, pts5)
            P = np.column_stack([axes[k][(gidx // (pts5[0] ** k)) % pts5[0]] for k in range(d5)])
            mo, vo = O.posterior_chol(P, ds5)
            em = max(np.max(np.abs(m[sel, i] - mo[:, i])) / max(np.max(np.abs(mo[:, i])), ds5["Y_std"][i]) for i in range(4))
            ev = max(np.max(np.abs(v[sel, i] - vo[:, i])) / (O.unpack_hyper(ds5["hypopt"][:, i], d5)[1] * ds5["Y_std"][i] ** 2) for i in range(4))
            out["posterior_parity_rank0_sample"] = {"points": 128, "mean_rel_err": float(em), "var_rel_err": float(ev), "tol": 1e-10,
                                                    "ok": bool(em <= 1e-10 and ev <= 1e-10)}
        eng.release(3)
        torch.cuda.empty_cache()
    except Exception as e:  # pragma: no cover
        out["error"] = repr(e)[:400]
    eng.set_option("fantasy_refine", int(args.refine))
    return out


DUMP_POINTS = 1 << 18      # per-point outputs are dumped at this many seeded points of the shard (all of a smaller one)
# step result fields -> the index field that is -1 when the reduction behind the value found no candidate
_INDEX_OF = {"best_value": "best_idx", "per_value": "per_idx", "undecided_best_value": "undecided_best_idx",
             "min_ucb0": "min_ucb0_idx", "min_lcb0": "min_lcb0_idx", "minimizer_var": "minimizer_idx",
             "target_lcb": "target_idx"}


class _DeviceF64:
    """A float64 device buffer of the library, exposed to torch through __cuda_array_interface__ (no copy; only read,
    but torch accepts no read-only flag)."""

    def __init__(self, ptr, shape):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": "<f8", "data": (int(ptr), False),
                                         "strides": None, "version": 3}


def dump_outputs(out_dir, eng, res, torch, dev):
    """--dump-outputs: what the last timed step computed, one DIR/<name>.npy per array.  The step's result as the
    caller receives it (sets, L, expander fields, x_new_idx; float64, nested keys joined by "_") and the per-point
    outputs the step leaves in the engine: posterior mean and variance (float64, (points, G) like GridEngine.posterior)
    and the safe / minimiser / unsafe masks (float32 0/1), at `point_index` (float64), a fixed seeded sample of
    DUMP_POINTS points of this rank's shard.  Under 40 MB in all (G <= 8).  The workloads are seeded, so two builds run
    with the same arguments can be compared array for array, except two work counters that were seen to vary between
    runs of one build (C4, 1 x B200): expander_n_ambiguous (pairs inside the TF32 error band, by one) and
    expander_pairs_evaluated (pairs the pruning keeps, by 2e-6 of them).
    A value whose index is -1 (no candidate) holds the library's +-inf sentinel; it is written as 0, as GridEngine
    already reports expander_std and minimizer_std, and the index says that it is absent."""
    from sbo_b200 import _capi as capi
    out = {}
    for k, v in res.items():
        scope, prefix = (v, k + "_") if isinstance(v, dict) else (res, "")
        for name in (v if isinstance(v, dict) else [k]):
            a = np.asarray(scope[name], dtype=np.float64)
            if _INDEX_OF.get(name) in scope:
                a = np.where(np.asarray(scope[_INDEX_OF[name]]) < 0, 0.0, a)
            out[prefix + name] = a
    cnt = eng.count
    sel = np.arange(cnt) if cnt <= DUMP_POINTS else np.sort(np.random.default_rng(0).choice(cnt, DUMP_POINTS, replace=False))
    out["point_index"] = sel.astype(np.float64)
    for name, kind in (("safe_mask", capi.MASK_SAFE), ("minimizer_mask", capi.MASK_MIN), ("unsafe_mask", capi.MASK_UNSAFE)):
        out[name] = eng.mask(kind)[sel].astype(np.float32)
    idx = torch.as_tensor(sel, device=dev)
    for name, ptr in zip(("posterior_mean", "posterior_var"), eng.posterior_dev()):
        buf = torch.as_tensor(_DeviceF64(ptr, (eng.G, cnt)), device=dev)          # [G][count], as the kernels write it
        out[name] = buf.index_select(1, idx).T.contiguous().cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_ours(args):
    import torch
    import torch.distributed as dist
    import sbo_b200
    from sbo_b200 import _capi as capi

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback (use --impl reference)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    (ds, lo, hi, pts, beta), wl_name = workload(args.workload)
    N = int(np.prod(pts))
    G = ds["Y_norm"].shape[1]
    n, d = ds["X_norm"].shape
    stream = torch.cuda.Stream(device=dev)
    eng = sbo_b200.GridEngine(local, stream=stream.cuda_stream)
    eng.set_grid(lo, hi, pts)
    if world > 1:
        eng.set_shard_cyclic(rank, world, 256)      # block-cyclic ownership balances |S| and |Z| over the ranks
        if args.orchestrator == "library":          # the library's own NCCL communicator: collectives inside the C ABI
            from sbo_b200 import sharded as _shc
            with torch.cuda.stream(stream):
                _shc.init_comm(eng, dev)
    fantasy = args.mode == "fantasy"
    eng.set_option("fantasy_prune", int(args.prune))
    eng.set_option("fantasy_refine", int(args.refine))

    def step(upload=True):
        """One acquisition step on this rank's shard.  Multi-GPU: collectives between the stages, issued on the
        engine's stream (torch's current stream inside this context) so they are ordered with its kernels."""
        with torch.cuda.stream(stream):
            if world == 1:
                return eng.safeopt_step(ds, beta, mode=args.mode, precision=args.precision, upload=upload)
            from sbo_b200 import sharded
            return sharded.safeopt_step(eng, ds, beta, mode=args.mode, precision=args.precision, upload=upload)

    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)   # 256 MiB > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-timed steps (value) ----
    clocks = Clocks(local)
    clocks.start()
    for _ in range(args.warmup):
        step()
    eng.kernel_launches(reset=True)
    barrier()
    clocks.mark()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    phases = []
    res = None
    for k in range(args.steps):
        flush.zero_()
        barrier()                      # ranks start every timed step together (no skew inside the event pair)
        with torch.cuda.stream(stream):
            ev[k][0].record(stream)
            res = step()
            ev[k][1].record(stream)
        phases.append(eng.phase_ms())
    barrier()
    clk = clocks.stop()
    launches = eng.kernel_launches()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, eng, res, torch, dev)
    ms = float(np.mean([a.elapsed_time(b) for a, b in ev]))
    # ---- end-to-end steps (host buffers in, host results out) ----
    t_e2e = []
    for k in range(args.e2e_steps if args.e2e_steps else max(2, args.steps)):
        flush.zero_()
        barrier()
        t0 = time.perf_counter()
        with torch.cuda.stream(stream):          # the collectives must be ordered with the engine's kernels
            r2 = step(upload=True)
            safe = eng.mask(capi.MASK_SAFE)
        torch.cuda.synchronize()
        t_e2e.append(time.perf_counter() - t0)
    e2e_s = float(np.mean(t_e2e[1:])) if len(t_e2e) > 1 else t_e2e[0]
    h2d = int(sum(np.asarray(ds[k]).nbytes for k in ("X_norm", "Y_norm", "X_mean", "X_std", "Y_mean", "Y_std", "hypopt")))
    d2h = int(safe.size // 8 + 512)
    if world > 1:
        t = torch.tensor([ms, e2e_s], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, e2e_s = float(t[0]), float(t[1])
    ex = res["expander"]
    # ---- the reference-exact (Lipschitz) acquisition steps on the same workload: SafeOpt and GoOSE step time ----
    lip = None
    if not args.no_lipschitz_steps:
        from sbo_b200 import sharded as _sh

        def lip_step(goose):
            with torch.cuda.stream(stream):
                if world == 1:
                    return eng.goose_step(ds, beta) if goose else eng.safeopt_step(ds, beta, mode="lipschitz", precision="fp64")
                return _sh.goose_step(eng, ds, beta) if goose else _sh.safeopt_step(eng, ds, beta, mode="lipschitz", precision="fp64")
        lip = {}
        for goose in (False, True):
            lip_step(goose)
            tl = []
            for _ in range(3):
                flush.zero_(); barrier()
                t0 = time.perf_counter(); rl = lip_step(goose); torch.cuda.synchronize(); tl.append(time.perf_counter() - t0)
            t = torch.tensor([float(np.mean(tl))], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            pr = rl["target"] if goose else rl["expander"]
            phl = eng.phase_ms()
            lip["goose" if goose else "safeopt"] = {"ms_per_step": float(t[0]) * 1e3, "phase_ms_rank0": {k: round(v, 3) for k, v in phl.items()},
                                                    "kernel_ms_rank0": round(sum(phl.values()), 3), "pairs": int(pr["pairs_algorithmic"]),
                                                    "pairs_evaluated": int(pr["pairs_evaluated"]), "n_hit": int(pr["n_hit"]),
                                                    "x_new_idx": int(rl["x_new_idx"])}
        lip["note"] = ("end-to-end wall time (host buffers) of one acquisition step with the reference's Lipschitz pair test "
                       "(SafeOpt.py:85-124, GoOSE.py:80-119), exact tile culling on; max over ranks")
    c5 = None
    if (args.c5 == 1 or (args.c5 < 0 and world == 8)) and args.workload == "c4":
        c5 = c5_key(args, eng, torch, dist, stream, rank, world, dev, barrier)
        eng.set_option("fantasy_refine", int(args.refine))
        eng.set_grid(lo, hi, pts)
        if world > 1:
            eng.set_shard_cyclic(rank, world, 256)
    pairs = int(ex["pairs_algorithmic"])            # sharded.safeopt_step already returns the global count
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    ph = {k: float(np.mean([p[k] for p in phases])) for k in phases[0]}     # rank 0's kernels
    peaks = {} if args.no_peaks else measure_peaks(torch, dev)
    mp = {}
    try:
        mp = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    # ---- roofline of the dominant kernel ----
    npad = ((n + 63) // 64) * 64
    if fantasy:
        # SURVEY 8d: F_exp = pairs*(2n + 3d + 20) per (x, z, constraint) pair-eval.  Only the pairs the kernel really
        # evaluates are charged (the exact pruning skips tile pairs that cannot hold a newly-safe pair); the split-TF32
        # mode issues 3 tensor passes for the same algorithmic GEMM, so `achieved` charges it ONE pass and
        # `tensor_tflops_issued` gives the rate the tensor pipe actually runs at.
        evaluated = int(ex["pairs_evaluated"])
        flops = evaluated / world * (2.0 * n + 3 * d + 20)      # rank 0's share (z is sharded evenly)
        t_k = ph["pairs"] * 1e-3
        passes = 3 if args.precision == "tf32x3" else 1
        t_k += ph.get("refine", 0.0) * 1e-3 * 0     # the FP64 refinement is its own phase (phase_ms.refine), not part of the GEMM
        if args.precision == "fp64":
            peak, src = peaks.get("fp64_tflops"), "cuBLAS FP64 GEMM measured in this run"
        elif mp.get("bf16_tflops_sustained"):
            # tcgen05 kind::tf32 runs at half the dense bf16 rate; the kernel runs ~0.5 s inside a long step, so the
            # sustained (power-capped) figure of MEASURED_PEAKS.json applies
            peak, src = mp["bf16_tflops_sustained"] / 2.0, "MEASURED_PEAKS.json bf16_tflops_sustained / 2 (TF32 = half the bf16 rate), of measured"
        else:
            peak, src = peaks.get("tf32_tflops"), "cuBLAS TF32 GEMM measured in this run (MEASURED_PEAKS.json absent)"
        roof = {"kernel": "tc::k_fantasy_tc2 (fantasy expander GEMM, 2-CTA tcgen05, %s)" % args.precision, "bound": "tensor",
                "achieved": flops / t_k / 1e12 if t_k > 0 else None,
                "peak": peak, "unit": "TFLOP/s", "traffic": TRAFFIC_NCU.get((args.workload, args.precision)),
                "peak_source": src, "cublas_tf32_tflops_this_run": peaks.get("tf32_tflops"),
                "algorithmic_flops_per_launch": flops, "kernel_ms": ph["pairs"],
                "tensor_passes": passes,
                "tensor_tflops_issued": (evaluated / world * 2.0 * n * passes) / t_k / 1e12 if t_k > 0 else None,
                "pairs_evaluated_fraction": evaluated / max(pairs, 1)}
    else:
        flops = float(G) * N / world * (float(n) * n + n * (3 * d + 6))     # SURVEY 8d F_post (per rank)
        t_k = (ph["solve"] + ph["crosscov"]) * 1e-3
        roof = {"kernel": "posterior solve (k_solve_var) + cross-covariance", "bound": "tensor",
                "achieved": flops / t_k / 1e12 if t_k > 0 else None, "peak": peaks.get("fp64_tflops"), "unit": "TFLOP/s",
                "traffic": None, "peak_source": "cuBLAS FP64 GEMM measured in this run (FP64 has no tcgen05 path)"}
    roof["frac"] = (roof["achieved"] / roof["peak"]) if roof.get("achieved") and roof.get("peak") else None
    value = pairs / (ms * 1e-3)
    line = {"metric": "expander_pair_evals_per_s", "value": value, "unit": "pair-evals/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": args.precision if (fantasy and args.precision != "fp64") else "f64",
            "data": "synthetic",
            "config": {"workload": wl_name, "mode": args.mode, "precision": args.precision, "N": N, "n": n, "d": d, "G": G,
                       "beta": beta, "n_safe": int(res["n_safe"]), "n_unsafe": int(res["n_unsafe"]), "n_min": int(res["n_min"]),
                       "pairs": pairs, "pairs_evaluated": int(ex["pairs_evaluated"]), "n_hit": int(ex["n_hit"]), "x_new_idx": int(res["x_new_idx"]),
                       "prune": int(args.prune), "refine": int(args.refine), "refined_pairs_fp64": int(ex.get("n_ambiguous", 0)), "refined_safe": int(ex.get("n_refined_safe", 0)), "n_undecided": int(ex.get("n_undecided", 0)),
                       "value_counts": "all |S|*|Z|*(G-1) pairs: the exact pruning decides the skipped ones without evaluating them",
                       "l2": "256 MiB flush buffer written between timed steps; working set >> L2",
                       "excludes": "plant evaluation and hyper-parameter fit (host side in the reference too)"},
            "value_evaluated_pairs_only": int(ex["pairs_evaluated"]) / (ms * 1e-3),
            "phase_ms": ph, "clocks": clk, "gpu_launches": int(launches // max(1, args.steps)),
            "e2e": {"value": pairs / e2e_s, "unit": "pair-evals/s", "ms_per_step": e2e_s * 1e3,
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "roofline": roof, "peaks": {**peaks, "hbm_gbs": mp.get("hbm_gbs"), "bf16_tflops": mp.get("bf16_tflops")}}
    if lip is not None:
        line["lipschitz_mode"] = lip
    if c5 is not None:
        if c5.get("pairs") and not args.no_cpu_baseline:       # the CPU arm on the same box, same model (bounded sample)
            from oracle import cpu_arm
            from sbo_b200 import workloads as _wl
            ds5, lo5, hi5, pts5, beta5 = _wl.c5()
            cores5 = use_all_host_threads()
            s5 = cpu_arm.sample_step(ds5, lo5, hi5, pts5, beta5, "fantasy", seed=0, n_points=8192, n_x=1024, n_z=16384)
            t5 = cpu_arm.extrapolate(s5, int(np.prod(pts5)), c5["pairs"])
            c5["cpu_baseline"] = {"value": c5["pairs"] / t5, "unit": "pair-evals/s", "cores": cores5, "kind": "port",
                                  "seconds_per_step_extrapolated": t5, "sample": cpu_arm.describe(s5, int(np.prod(pts5)), c5["pairs"], "fantasy")}
            c5["speedup_vs_cpu_port"] = t5 / (c5["ms_per_step"] * 1e-3)
        line["c5"] = c5
    if world == 1 and not args.no_reference_configs:
        line["reference_configs"] = reference_configs(eng, torch)
    if not args.no_cpu_baseline and world == 1:
        from oracle import cpu_arm
        cpu_threads = use_all_host_threads()
        s = cpu_arm.sample_step(ds, lo, hi, pts, beta, args.mode, seed=0, **CPU_BASELINE_SAMPLE)
        t_full = cpu_arm.extrapolate(s, N, pairs)
        line["cpu_baseline"] = {"value": pairs / t_full, "unit": "pair-evals/s", "cores": cpu_threads, "kind": "port",
                                "ms_per_step_extrapolated": t_full * 1e3,
                                "pair_stage_pair_evals_per_s": s["pairs"] / s["t_pairs"] if s["t_pairs"] > 0 else None,
                                "sample": cpu_arm.describe(s, N, pairs, args.mode)}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
