"""Multi-GPU acquisition steps: one process per GPU, the grid sharded block-cyclically over the ranks
(SURVEY.md section 8e).  Every rank runs the same kernels on its shard through its own ``GridEngine``;
this module only inserts the collectives (``torch.distributed``: NCCL on GPUs, gloo in the CPU tests):

  all-reduce-min  (min_S ucb_0, index) and (min_S lcb_0, index)      between the two set passes
  all-reduce-max  Lipschitz constants, (max_M var_0, index)
  broadcasts      the candidates' rows (+ V rows in fantasy mode), one block per rank straight into the gathered
                  buffer (an all-gather with uneven blocks): every rank pairs ALL candidates x in S with ITS OWN
                  unsafe points z
  all-reduce      per-candidate hit flags (max) / newly-safe counts (sum); none for the fantasy GoOSE target, whose
                  verdict on an unsafe point is local
  all-gather      local optima (value, global index) -> deterministic reduction, lowest index on ties

The engine is any object with the GridEngine staged-pair interface, so the orchestration is testable on CPU
with a NumPy stand-in (tests/test_sharded_gloo.py).
"""
from __future__ import annotations

import numpy as np
import torch
import torch.distributed as dist

from . import _capi as capi


# ---------------------------------------------------------------------------------------------
# library-owned communicator (csrc/comm.cu): torch.distributed only carries the 128-byte NCCL id to the ranks
# ---------------------------------------------------------------------------------------------
def init_comm(eng, device=None, group=None):
    """Create the library's own NCCL communicator over the ranks of `group`; afterwards safeopt_step / goose_step run
    with every collective inside the library (sbo_safeopt_step_sharded / sbo_goose_step_sharded)."""
    device = torch.device("cuda", eng.device) if device is None else device
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    t = torch.zeros(128, dtype=torch.uint8, device=device)
    if rank == 0:
        t.copy_(torch.frombuffer(bytearray(eng.comm_unique_id()), dtype=torch.uint8))
    dist.broadcast(t, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
    eng.comm_init(rank, world, bytes(t.cpu().numpy().tobytes()))


# ---------------------------------------------------------------------------------------------
# small collectives
# ---------------------------------------------------------------------------------------------
def _sync(device):
    if device.type == "cuda":
        torch.cuda.synchronize(device)


def _order(eng, device):
    """Order the engine's kernels with torch's collectives: nothing to do when both use the same CUDA stream
    (bench.py runs the step inside torch.cuda.stream(engine stream)), else a device synchronise."""
    if device.type != "cuda":
        return
    if getattr(eng, "stream", None) is not None and eng.stream == torch.cuda.current_stream(device).cuda_stream:
        return
    torch.cuda.synchronize(device)


def gather_scalars(values, device, group=None):
    """all-gather a short list of python floats -> (world, len) float64 numpy array."""
    world = dist.get_world_size(group)
    t = torch.tensor([float(v) for v in values], dtype=torch.float64, device=device)
    out = torch.empty(world * t.numel(), dtype=torch.float64, device=device)
    dist.all_gather_into_tensor(out, t, group=group)           # flat in / flat out: accepted by NCCL and gloo
    return out.view(world, t.numel()).cpu().numpy()


def reduce_arg(pairs, device, maximize=False, group=None):
    """pairs = [(value, global_index), ...] local optima (index -1 = empty).  Returns the global optimum of each
    pair over all ranks: best value, lowest index on ties; (+-inf, -1) if every rank is empty."""
    flat = []
    for v, i in pairs:
        flat += [float(v), float(i)]
    g = gather_scalars(flat, device, group)          # indices < 2^53 are exact in float64
    out = []
    for k in range(len(pairs)):
        vals, idxs = g[:, 2 * k], g[:, 2 * k + 1].astype(np.int64)
        ok = idxs >= 0
        if not ok.any():
            out.append((-np.inf if maximize else np.inf, -1))
            continue
        v = np.where(ok, vals, -np.inf if maximize else np.inf)
        best = v.max() if maximize else v.min()
        cand = idxs[ok & (v == best)]
        out.append((float(best), int(cand.min())))
    return out


def exchange_rows(buf, n_all, group=None):
    """buf (sum n_r, w) already holds THIS rank's rows at its offset; fill in every other rank's block in place.
    One broadcast per non-empty rank straight into the destination slice: no padding, no concatenation copy
    (the V rows are 41 GB at C5), and uneven block sizes cost nothing."""
    off = 0
    for r, n in enumerate(n_all):
        n = int(n)
        if n:
            dist.broadcast(buf[off: off + n], src=dist.get_global_rank(group, r) if group is not None else r, group=group)
        off += n
    return buf


class _Trace:
    """SBO_SHARDED_TRACE=1: rank 0 prints the wall time of every stage (device-synchronised) -- diagnosis only."""

    def __init__(self, device):
        import os
        self.on = os.environ.get("SBO_SHARDED_TRACE") == "1"
        self.device, self.t, self.rows = device, None, []

    def mark(self, name):
        if not self.on:
            return
        import time
        _sync(self.device)
        now = time.perf_counter()
        if self.t is not None:
            self.rows.append((name, (now - self.t) * 1e3))
        self.t = now

    def dump(self):
        if self.on and dist.get_rank() == 0:
            print("sharded trace (ms): " + "  ".join(f"{n}={t:.2f}" for n, t in self.rows), flush=True)


def first_best(per_value, per_idx, maximize):
    """SafeOpt.py:120-122 / GoOSE.py:110-112: python max()/min() keep the FIRST optimum over the constraints."""
    bi, bv = -1, (-np.inf if maximize else np.inf)
    for v, i in zip(per_value, per_idx):
        if i >= 0 and (bi < 0 or (v > bv if maximize else v < bv)):
            bi, bv = i, v
    return bi, bv


# ---------------------------------------------------------------------------------------------
# stages shared by the SafeOpt and GoOSE steps
# ---------------------------------------------------------------------------------------------
def _posterior_and_sets(eng, ds, beta, unsafe_rule, with_grad, keep_v, upload, device, group, need_pass2=True, kernel="RBF"):
    if upload:
        if kernel == "RBF":
            eng.set_model(ds)             # the one-argument form keeps engines that only know the SE kernel usable here
        else:
            eng.set_model(ds, kernel)
    eng.posterior(with_grad=with_grad, keep_v=keep_v, fetch=False)
    s1 = eng.sets_pass1(beta, unsafe_rule)
    (min_ucb0, min_ucb0_idx), (min_lcb0, min_lcb0_idx) = reduce_arg(
        [(s1["min_ucb0"], s1["min_ucb0_idx"]), (s1["min_lcb0"], s1["min_lcb0_idx"])], device, False, group)
    out = {"min_ucb0": min_ucb0, "min_ucb0_idx": min_ucb0_idx, "min_lcb0": min_lcb0, "min_lcb0_idx": min_lcb0_idx}
    n_min = 0
    if need_pass2:
        s2 = eng.sets_pass2(min_ucb0)
        (mv, mi), = reduce_arg([(s2["minimizer_var"], s2["minimizer_idx"])], device, True, group)
        out.update({"minimizer_var": mv, "minimizer_idx": mi})
        n_min = s2["n_min"]
    tot = gather_scalars([s1["n_safe"], s1["n_unsafe"], n_min], device, group).sum(axis=0)
    out.update({"n_safe": int(tot[0]), "n_unsafe": int(tot[1]), "n_min": int(tot[2])})
    if with_grad:
        out["L"] = gather_scalars(list(eng.lipschitz()), device, group).max(axis=0)
    return out


BIG_V_BYTES = 4 << 30      # above this the per-point V rows and the gathered copies are released as soon as possible


def _pairs(eng, mode, prec, beta, L, goose, device, group, want_counts=False):
    """prepare -> export into the gathered buffer -> broadcast blocks -> import -> run -> all-reduce -> finish ->
    reduce the local optima."""
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    tr = _Trace(device)
    tr.mark("start")
    info = eng.pairs_prepare(mode, prec, beta, L)
    nx, nz = int(info["n_x_local"]), int(info["n_z_local"])
    n_all = gather_scalars([nx], device, group)[:, 0].astype(np.int64)
    n_total, offset = int(n_all.sum()), int(n_all[:rank].sum())
    fantasy = mode == capi.MODE_FANTASY
    if fantasy and not goose and world > 1 and getattr(eng, "options", {}).get("fantasy_refine") == 3:
        raise ValueError("fantasy_refine = 3 (bounds mode) on several ranks needs the library communicator: "
                         "init_comm() / orchestrator='library' (the per-candidate undecided counts are combined there)")
    if not fantasy and world > 1 and hasattr(eng, "pairs_set_segments"):
        # reference-exact mode: the library restores grid order of the gathered candidates (compact tiles for the exact
        # culling), and the SafeOpt expander is split by CANDIDATES: all-gather of the unsafe bitmask (north_star's
        # collective; N/8 bytes in total), every rank pairs its share of the candidate tiles with ALL unsafe points
        eng.pairs_set_segments(n_all, rank)
        if not goose:
            wpr = int(gather_scalars([(eng.count + 31) // 32], device, group)[:, 0].max())
            loc = torch.zeros(wpr, dtype=torch.int32, device=device)
            eng.mask_export(capi.MASK_UNSAFE, loc)
            allw = torch.empty(world * wpr, dtype=torch.int32, device=device)
            _order(eng, device)
            dist.all_gather_into_tensor(allw, loc, group=group)
            _order(eng, device)
            eng.pairs_set_global_unsafe(allw, wpr, world)
    tr.mark("prepare")
    vrow = int(info["vrow_bytes"])
    big = vrow * n_total > BIG_V_BYTES
    rows_all = torch.empty((max(n_total, 1), int(info["row_doubles"])), dtype=torch.float64, device=device)
    v_all = torch.empty((max(n_total, 1), max(vrow, 1)), dtype=torch.uint8, device=device) if vrow else None
    # every rank writes its candidates' rows straight into its slice of the gathered buffers
    eng.pairs_export(rows_all[offset: offset + max(nx, 1)] if nx else rows_all,
                     (v_all[offset: offset + max(nx, 1)] if nx else v_all) if vrow else None)
    if big and hasattr(eng, "release"):
        eng.release(1)                       # the per-point V rows are not needed after the export
    tr.mark("export")
    _order(eng, device)
    exchange_rows(rows_all, n_all, group)
    if vrow:
        exchange_rows(v_all, n_all, group)
    tr.mark("exchange")
    _order(eng, device)
    eng.pairs_import(n_total, rows_all, v_all)
    if big:
        _sync(device)
        del v_all
        v_all = None
        if device.type == "cuda":
            torch.cuda.empty_cache()         # hand the gathered copy back before the GEMM workspaces are sized
    tr.mark("import")
    nc = eng.G - 1
    if goose and fantasy:                  # hit words over this rank's prepared unsafe slots
        result = torch.zeros(max((nz + 31) // 32, 1), dtype=torch.int32, device=device)
    elif goose:
        result = torch.zeros(max(nc * nz, 1), dtype=torch.uint8, device=device)
    elif fantasy:
        result = torch.zeros(max(n_total, 1), dtype=torch.int32, device=device)
    else:
        result = torch.zeros(max(nc * n_total, 1), dtype=torch.uint8, device=device)
    _order(eng, device)
    eng.pairs_run(goose, result)
    tr.mark("run")
    _order(eng, device)
    if not goose and n_total > 0:          # x is global: combine the verdicts of all z shards
        dist.all_reduce(result, op=dist.ReduceOp.SUM if fantasy else dist.ReduceOp.MAX, group=group)
    tr.mark("allreduce")
    _order(eng, device)
    loc = eng.pairs_finish(goose, 0 if goose else offset, result, want_counts=want_counts)
    nmask = 1 if fantasy else nc
    red = reduce_arg([(loc["per_value"][c], loc["per_idx"][c]) for c in range(nmask)], device, not goose, group) if nmask else []
    per_value, per_idx = [v for v, _ in red], [i for _, i in red]
    bi, bv = first_best(per_value, per_idx, maximize=not goose)
    tot = gather_scalars([nz, loc["n_hit"], loc["pairs_evaluated"], loc.get("n_ambiguous", 0), loc.get("n_refined_safe", 0)],
                         device, group).sum(axis=0)
    if big and hasattr(eng, "release"):
        eng.release(2)                       # gathered operands: the next step's V rows need the room
    tr.mark("finish")
    tr.dump()
    out = {"best_idx": bi, "best_value": bv, "per_idx": per_idx, "per_value": per_value, "n_x": n_total,
           "n_z": int(tot[0]), "n_hit": int(tot[1]), "pairs_evaluated": int(tot[2]),
           "pairs_algorithmic": n_total * int(tot[0]) * nc, "n_ambiguous": int(tot[3]), "n_refined_safe": int(tot[4]), "local": loc}
    if goose and fantasy:                  # bounds mode: the undecided unsafe points are local too
        (uv, ui), = reduce_arg([(loc.get("undecided_best_value", np.inf), loc.get("undecided_best_idx", -1))], device, False, group)
        out.update({"n_undecided": int(gather_scalars([loc.get("n_undecided", 0)], device, group).sum()),
                    "undecided_best_idx": ui, "undecided_best_value": uv})
    return out


# ---------------------------------------------------------------------------------------------
# whole steps (same decision rules as GridEngine.safeopt_step / goose_step)
# ---------------------------------------------------------------------------------------------
def safeopt_step(eng, ds, beta, mode="lipschitz", precision="fp64", unsafe_rule=capi.UNSAFE_ALL, L=None, upload=True,
                 device=None, group=None, kernel="RBF"):
    """test/test_SafeOpt.py:144-158 on a sharded grid.  Every rank returns the same global result."""
    if getattr(eng, "comm_ready", False) and group is None:
        return eng.safeopt_step_sharded(ds, beta, mode=mode, precision=precision, unsafe_rule=unsafe_rule, L=L, upload=upload,
                                        kernel=kernel)
    device = torch.device("cuda", eng.device) if device is None else device
    fantasy = mode == "fantasy"
    prec, kv = capi.PRECISIONS[precision]
    out = _posterior_and_sets(eng, ds, beta, unsafe_rule, with_grad=(not fantasy and L is None),
                              keep_v=kv if fantasy else 0, upload=upload, device=device, group=group, kernel=kernel)
    out["minimizer_std"] = float(np.sqrt(out["minimizer_var"])) if out["minimizer_idx"] >= 0 else 0.0
    if fantasy:
        ex = _pairs(eng, capi.MODE_FANTASY, prec, beta, None, False, device, group)
    else:
        if L is None:
            L = np.full(eng.G, out["L"][eng.G - 1])              # SafeOpt.py:110
        ex = _pairs(eng, capi.MODE_LIPSCHITZ, capi.PREC_FP64, beta, L, False, device, group)
    out["expander"] = ex
    out["expander_idx"] = ex["best_idx"]
    out["expander_std"] = float(np.sqrt(ex["best_value"])) if ex["best_idx"] >= 0 else 0.0
    out["x_new_idx"] = out["minimizer_idx"] if out["minimizer_std"] > out["expander_std"] else ex["best_idx"]
    return out


def goose_step(eng, ds, beta, unsafe_rule=capi.UNSAFE_ALL, L=None, upload=True, device=None, group=None, coords=None,
               mode="lipschitz", precision="fp64", kernel="RBF"):
    """test/test_GoOSE.py:151-162 on a sharded grid.  mode="fantasy": candidate and V rows are exchanged as in the
    SafeOpt fantasy step, then every rank decides its own unsafe points (no result all-reduce)."""
    if getattr(eng, "comm_ready", False) and group is None:
        return eng.goose_step_sharded(ds, beta, unsafe_rule=unsafe_rule, L=L, upload=upload, mode=mode, precision=precision,
                                      kernel=kernel)
    device = torch.device("cuda", eng.device) if device is None else device
    fantasy = mode == "fantasy"
    prec, kv = capi.PRECISIONS[precision]
    out = _posterior_and_sets(eng, ds, beta, unsafe_rule, with_grad=(not fantasy and L is None), keep_v=kv if fantasy else 0,
                              upload=upload, device=device, group=group, need_pass2=False, kernel=kernel)
    if fantasy:
        tg = _pairs(eng, capi.MODE_FANTASY, prec, beta, None, True, device, group)
    else:
        if L is None:
            L = np.full(eng.G, out["L"][eng.G - 1])              # GoOSE.py:100
        tg = _pairs(eng, capi.MODE_LIPSCHITZ, capi.PREC_FP64, beta, L, True, device, group)
    out["target"] = tg
    out["target_idx"], out["target_lcb"] = tg["best_idx"], tg["best_value"]
    if out["min_lcb0"] <= tg["best_value"] or tg["best_idx"] < 0:
        out["x_new_idx"], out["explore_idx"] = out["min_lcb0_idx"], -1
    else:
        target = eng.point_coords(tg["best_idx"])
        li, ld = eng.argreduce(capi.ARGMIN_DIST, capi.MASK_SAFE, 0, target)
        (d, i), = reduce_arg([(ld, li)], device, False, group)
        out["x_new_idx"] = out["explore_idx"] = i
    return out


def safeopt_batch(eng, q, device=None, group=None):
    """Batch SafeOpt acquisition (GridEngine.safeopt_batch) on a sharded grid, after a SafeOpt step of this module on every
    rank: per pick each rank reports its local optima over M and E, the ranks agree on the global ones (largest std, lowest
    index on ties) and apply the pick rule, and every rank hallucinates the same observation.  Every rank returns the same
    list of picks."""
    if getattr(eng, "comm_ready", False) and group is None:
        return eng.safeopt_batch_sharded(q)
    device = torch.device("cuda", eng.device) if device is None else device
    eng.batch_prepare(q)
    picks = []
    for b in range(int(q)):
        loc = eng.batch_local()
        (sm, im), (se, ie) = reduce_arg([(loc["std_min"], loc["idx_min"]), (loc["std_exp"], loc["idx_exp"])], device, True, group)
        sm, se = (sm if im >= 0 else 0.0), (se if ie >= 0 else 0.0)
        take_min = im >= 0 and (ie < 0 or sm > se)                 # test/test_SafeOpt.py:153-158, an empty set yields
        idx = im if take_min else ie
        if idx < 0:                                                # M and E are empty on every rank, and stay so
            break
        picks.append({"idx": idx, "from_expander": 0 if take_min else 1, "std_min": sm, "idx_min": im, "std_exp": se, "idx_exp": ie})
        if b + 1 < q:
            eng.batch_commit(idx)
    return picks


def goose_batch(eng, q, device=None, group=None):
    """Batch GoOSE acquisition (GridEngine.goose_batch) on a sharded grid, after a GoOSE step of this module on every rank:
    per pick each rank reports its local optima of lcb_0 over S_b and T_b, the ranks agree on the global ones (smallest,
    lowest index on ties) and apply the rule of test/test_GoOSE.py:158-162; an explore pick takes the globally nearest
    remaining safe point to the target.  Every rank hallucinates the same observation and returns the same picks."""
    if getattr(eng, "comm_ready", False) and group is None:
        return eng.goose_batch_sharded(q)
    device = torch.device("cuda", eng.device) if device is None else device
    eng.goose_batch_prepare(q)
    picks = []
    for b in range(int(q)):
        loc = eng.goose_batch_local()
        (sl, si), (tl, ti) = reduce_arg([(loc["safe_lcb"], loc["safe_idx"]), (loc["target_lcb"], loc["target_idx"])], device, False, group)
        if si < 0:                                                 # S_b is empty on every rank, and stays so
            break
        explore = ti >= 0 and not sl <= tl                         # test/test_GoOSE.py:158-162
        idx, dist = si, 0.0
        if explore:
            (d2, idx), = reduce_arg([eng.goose_batch_nearest(ti)[::-1]], device, False, group)
            dist = float(np.sqrt(d2))
        picks.append({"idx": idx, "explore": int(explore), "safe_lcb": sl, "safe_idx": si, "target_lcb": tl, "target_idx": ti,
                      "dist": dist})
        if b + 1 < q:
            eng.goose_batch_commit(idx, ti if explore else -1)
    return picks
