"""Several ranks of the sharded step on one GPU: W host threads, each with its own GridEngine (its own sbo_ctx on cuda:0)
on its rotated block-cyclic shard, exchange through in-process stand-ins for the torch.distributed collectives that
sbo_b200.sharded calls.  The kernels and the orchestration are then exactly those of a torch-orchestrated multi-GPU run,
so the code that only runs with more than one rank is checked on one GPU:

  export / import of the candidates with their global grid index (and V rows), the fantasy key sort over all candidates,
  grid order restored from the rank-major segments (k_canon_perm), the global unsafe mask rebuilt from the ranks' local
  masks (k_assemble_global_mask), candidate tiles dealt to the ranks, results read out at each rank's offset, the FP64
  refinement of pairs whose candidate belongs to another rank, and the fantasy GoOSE target over each rank's own z.

Every case compares the reassembled per-rank masks and counts with one unsharded context and with the FP64 oracle, and
asserts that the edge it is there for actually occurs on the GPU's own sets.  The harness itself is checked on the CPU
against the oracle step with the NumPy stand-in engine of test_sharded_gloo.py."""
import threading
import time
import types

import numpy as np
import pytest
import torch
import torch.distributed as tdist

from conftest import golden_ds, load_golden
from goose_fantasy_ref import goose_target_fantasy
from test_sharded_gloo import OracleEngine

RANK_TIMEOUT = 300.0         # seconds a rank may wait at a collective, and the main thread for all ranks
FANTASY_PRECISIONS = ("fp64", "tf32", "tf32x3")
TARGET_PRECISIONS = ("fp64", "tf32")
EXACT_TOL = 1e-12            # tests/test_gpu_parity.py _fantasy_tc_case: refined decisions are the FP64 ones outside this band


# ---------------------------------------------------------------------------------------------------------------------
# in-process collectives: one ThreadComm per run, group handle = (comm, rank)
# ---------------------------------------------------------------------------------------------------------------------
class ThreadComm:
    def __init__(self, world, timeout=RANK_TIMEOUT):
        self.world = world
        self.barrier = threading.Barrier(world, timeout=timeout)
        self.slots = [None] * world


def _exchange(group, t):
    """Deposit a copy of t, wait for every rank, read all deposits, wait again (so that no rank replaces its deposit
    before the others have read it).  The device is synchronised first: the engine may have written t on its own stream."""
    comm, rank = group
    if t.is_cuda:
        torch.cuda.synchronize(t.device)
    comm.slots[rank] = t.detach().to("cpu", copy=True)
    comm.barrier.wait()
    vals = list(comm.slots)
    comm.barrier.wait()
    return vals


def _store(t, value):
    t.copy_(value.reshape(t.shape).to(device=t.device, dtype=t.dtype))
    if t.is_cuda:
        torch.cuda.synchronize(t.device)


def _group(group):
    assert group is not None, "pass group= so that the sharded steps take the torch.distributed path"
    return group


def _broadcast(t, src, group=None):
    _store(t, _exchange(_group(group), t)[src])


def _all_gather_into_tensor(out, t, group=None):
    vals = _exchange(_group(group), t)
    _store(out, torch.cat([v.reshape(-1) for v in vals]))


def _all_reduce(t, op=tdist.ReduceOp.SUM, group=None):
    s = torch.stack(_exchange(_group(group), t))
    if op == tdist.ReduceOp.SUM:
        _store(t, s.sum(0))
    elif op == tdist.ReduceOp.MAX:
        _store(t, s.amax(0))
    else:
        raise NotImplementedError(f"reduce op {op}")


THREAD_DIST = types.SimpleNamespace(
    ReduceOp=tdist.ReduceOp,
    get_rank=lambda group=None: _group(group)[1],
    get_world_size=lambda group=None: _group(group)[0].world,
    get_global_rank=lambda group, r: r,
    broadcast=_broadcast,
    all_gather_into_tensor=_all_gather_into_tensor,
    all_reduce=_all_reduce,
)


@pytest.fixture
def sharded(monkeypatch):
    import sbo_b200  # noqa: F401
    from sbo_b200 import sharded as mod
    monkeypatch.setattr(mod, "dist", THREAD_DIST)
    return mod


def run_ranks(world, make_engine, body, timeout=RANK_TIMEOUT):
    """One thread per rank: eng = make_engine(rank, world); result = body(eng, rank, group); the engine is closed in the
    same thread.  A rank that raises aborts the barrier, so the others fail at their next collective instead of waiting;
    the first error is raised here.  Returns the per-rank results."""
    comm = ThreadComm(world, timeout)
    results, errors = [None] * world, [None] * world

    def main(rank):
        eng = None
        try:
            eng = make_engine(rank, world)
            results[rank] = body(eng, rank, (comm, rank))
        except BaseException as e:          # noqa: B902 -- re-raised by the main thread
            errors[rank] = e
            comm.barrier.abort()
        finally:
            if eng is not None and hasattr(eng, "close"):
                eng.close()

    threads = [threading.Thread(target=main, args=(r,), name=f"rank{r}") for r in range(world)]
    for t in threads:
        t.start()
    deadline = time.monotonic() + timeout
    for t in threads:
        t.join(max(0.0, deadline - time.monotonic()))
    hung = [t.name for t in threads if t.is_alive()]
    if hung:
        comm.barrier.abort()
        for t in threads:
            t.join(60.0)
    errs = [e for e in errors if e is not None]
    first = next((e for e in errs if not isinstance(e, threading.BrokenBarrierError)), errs[0] if errs else None)
    if first is not None:
        raise first
    assert not hung, f"ranks still running after {timeout} s: {hung}"
    return results


def shard_gidx(rank, world, N, block):
    """Global grid index of every local point of `rank` (rotated block-cyclic, sbo_set_shard_cyclic)."""
    return OracleEngine.shard_gidx(rank, world, N, block)


def to_global(local, world, N, block, dtype=None):
    """Per-rank local arrays -> one array in grid order; the shards must tile the grid."""
    out = np.zeros(N, dtype=dtype or np.asarray(local[0]).dtype)
    seen = np.zeros(N, dtype=np.int64)
    for r in range(world):
        g = shard_gidx(r, world, N, block)
        assert len(local[r]) == g.size, (r, len(local[r]), g.size)
        out[g] = local[r]
        seen[g] += 1
    assert (seen == 1).all()
    return out


def _record_prepare(eng):
    """Keep what every pairs_prepare of this engine reported (n_x_local, n_z_local: the rank's own sets)."""
    infos, prepare = [], eng.pairs_prepare

    def wrapped(*args, **kw):
        info = prepare(*args, **kw)
        infos.append(info)
        return info
    eng.pairs_prepare = wrapped
    return infos


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the harness against the single-process oracle step (NumPy stand-in engine, no kernel)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("world", [3, 8])
@pytest.mark.parametrize("case", [
    {"gold": "c3_wor", "n": 35, "beta": 2.0, "grid": [29, 23], "mode": "lipschitz", "rule": "all"},
    {"gold": "c1_benoit", "n": 9, "beta": 3.0, "grid": [36, 30], "mode": "lipschitz", "rule": "any"},
    {"gold": "c1_benoit", "n": 9, "beta": 3.0, "grid": [40, 36], "mode": "fantasy", "rule": "all"},
    {"gold": "c3_wor", "n": 20, "beta": 2.0, "grid": [22, 19], "mode": "fantasy", "rule": "any"},
])
def test_thread_ranks_reproduce_the_oracle_step(sharded, oracle, case, world):
    gold = load_golden(case["gold"])
    ds = golden_ds(oracle, gold, case["n"])
    beta, lip, rule = case["beta"], case["mode"] == "lipschitz", case["rule"]
    rid = 1 if rule == "any" else 0                     # sbo_b200._capi.UNSAFE_ANY / UNSAFE_ALL
    dev = torch.device("cpu")

    def make(rank, w):
        return OracleEngine(oracle, rank, w, gold["lo"], gold["hi"], case["grid"])

    def body(eng, rank, g):
        st = sharded.safeopt_step(eng, ds, beta, mode=case["mode"], unsafe_rule=rid, device=dev, group=g)
        out = {k: st[k] for k in ("n_safe", "n_unsafe", "n_min", "minimizer_idx", "expander_idx", "x_new_idx", "min_ucb0")}
        out["n_hit"] = st["expander"]["n_hit"]
        out["n_x"] = st["expander"]["n_x"]
        if lip:
            gs = sharded.goose_step(eng, ds, beta, unsafe_rule=rid, device=dev, group=g)
            out.update({"g_" + k: gs[k] for k in ("min_lcb0_idx", "target_idx", "x_new_idx", "explore_idx")})
        return out

    res = run_ranks(world, make, body)
    assert all(r == res[0] for r in res)
    pts = oracle.make_grid(gold["lo"], gold["hi"], case["grid"])
    so = oracle.safeopt_step(pts, ds, beta, mode=case["mode"], unsafe_rule=rule, form="chol")
    r = res[0]
    assert (r["n_safe"], r["n_unsafe"], r["n_min"]) == (so["S"].sum(), so["Z"].sum(), so["M"].sum())
    assert r["n_x"] == so["S"].sum()
    assert (r["minimizer_idx"], r["expander_idx"], r["x_new_idx"]) == (so["minimizer_idx"], so["expander_idx"], so["x_new_idx"])
    assert r["min_ucb0"] == pytest.approx(so["min_ucb0"], rel=1e-12)
    assert r["n_hit"] == np.any(so["expander_masks"], axis=0).sum() > 0
    if lip:
        go = oracle.goose_step(pts, ds, beta, unsafe_rule=rule, form="chol")
        assert (r["g_min_lcb0_idx"], r["g_target_idx"]) == (go["safe_min_idx"], go["target_idx"])
        assert (r["g_x_new_idx"], r["g_explore_idx"]) == (go["x_new_idx"], go["explore_idx"])


def test_a_failing_rank_fails_the_run_without_hanging(sharded):
    """The rank that raises is reported; the ranks waiting at a collective are released by the aborted barrier."""
    def body(eng, rank, g):
        if rank == 1:
            raise RuntimeError("rank 1 failed")
        sharded.gather_scalars([rank], torch.device("cpu"), g)

    t0 = time.monotonic()
    with pytest.raises(RuntimeError, match="rank 1 failed"):
        run_ranks(3, lambda rank, world: None, body)
    assert time.monotonic() - t0 < RANK_TIMEOUT / 2
    assert not [t for t in threading.enumerate() if t.name.startswith("rank")]


def test_thread_collectives(sharded):
    dev = torch.device("cpu")

    def body(eng, rank, g):
        d = sharded.dist
        s = torch.tensor([rank, 10 * rank], dtype=torch.int32)
        d.all_reduce(s, op=d.ReduceOp.SUM, group=g)
        m = torch.tensor([rank, 3 - rank], dtype=torch.uint8)
        d.all_reduce(m, op=d.ReduceOp.MAX, group=g)
        f = torch.tensor([0.5 * rank], dtype=torch.float64)
        d.all_reduce(f, op=d.ReduceOp.MAX, group=g)
        b = torch.arange(4, dtype=torch.float64) + 100 * rank
        d.broadcast(b[1:3], src=2, group=g)                    # into a slice, as sharded.exchange_rows does
        ga = sharded.gather_scalars([rank, -rank], dev, g)
        return s.tolist(), m.tolist(), f.tolist(), b.tolist(), ga.tolist()

    res = run_ranks(3, lambda rank, world: None, body)
    for rank, (s, m, f, b, ga) in enumerate(res):
        assert s == [3, 30] and m == [2, 3] and f == [1.0]
        assert b == [100 * rank, 201.0, 202.0, 100 * rank + 3]
        assert ga == [[0, 0], [1, -1], [2, -2]]


# ---------------------------------------------------------------------------------------------------------------------
# GPU cases
# ---------------------------------------------------------------------------------------------------------------------
# name -> (workload, edge).  Golden workloads: (gold, n, beta, grid, rule); synthetic: workloads.small arguments
CASES = {
    # N = 2745 is not a multiple of the block; the last super-block is partial at 3 and 8 ranks and the ranks' mask word
    # counts differ there (zero padding in k_assemble_global_mask)
    "c3_ragged": {"gold": ("c3_wor", 20, 2.0, [45, 61], "any")},
    # ranks without candidates next to ranks with some
    "c1_ranks_without_candidates": {"gold": ("c1_benoit", 4, 3.0, [64, 64], "all")},
    # ranks without unsafe points next to ranks with some
    "c3_ranks_without_unsafe": {"gold": ("c3_wor", 35, 2.0, [64, 64], "all")},
    # no candidate on any rank
    "c1_empty_safe_set": {"gold": ("c1_benoit", 4, 500.0, [64, 64], "all")},
    # a non-SE covariance function must reach every rank
    "matern52": {"small": dict(d=3, pts_per_dim=14, n=70, seed=23, G=3), "rule": "all", "kernel": "Matern52"},
    # npad = 256, three constraints: the FP64 refinement cut into cells and re-run after a list overflow
    "small_d4": {"small": dict(d=4, pts_per_dim=9, n=200, seed=24, G=4), "rule": "any"},
}
LAYOUTS = [("c3_ragged", 2, 32), ("c3_ragged", 3, 32), ("c3_ragged", 8, 32), ("c1_ranks_without_candidates", 8, 256),
           ("c3_ranks_without_unsafe", 8, 256), ("c1_empty_safe_set", 3, 32), ("matern52", 3, 32)]
_REF = {}                    # references per (kind, case): computed once, reused across world sizes


def _capi():
    from sbo_b200 import _capi
    return _capi


def _rule_id(rule):
    capi = _capi()
    return capi.UNSAFE_ANY if rule == "any" else capi.UNSAFE_ALL


def _workload(oracle, name):
    """(ds, lo, hi, grid, beta, rule, kernel) of a case."""
    c = CASES[name]
    if "gold" in c:
        gname, n, beta, grid, rule = c["gold"]
        gold = load_golden(gname)
        return golden_ds(oracle, gold, n), gold["lo"], gold["hi"], grid, beta, rule, "RBF"
    from sbo_b200 import workloads
    ds, lo, hi, pts, beta = workloads.small(**c["small"])
    return dict(ds), lo, hi, pts, beta, c["rule"], c.get("kernel", "RBF")


def _gpu_engines(lo, hi, grid, block, options=()):
    def make(rank, world):
        import sbo_b200
        eng = sbo_b200.GridEngine(0)
        try:
            eng.set_grid(lo, hi, grid)
            eng.set_shard_cyclic(rank, world, block)
            for k, v in options:
                eng.set_option(k, v)
        except BaseException:
            eng.close()
            raise
        return eng
    return make


def _assert_edge(name, world, block, N, counts, nx, nz):
    """The edge a case is there for, on the GPU's own sets (n_x_local / n_z_local of each rank's pairs_prepare)."""
    nblk = -(-N // block)
    assert N >= world * block and all(c > 0 for c in counts)
    if name == "c3_ragged":
        assert N % block != 0
        if world > 2:
            words = {(c + 31) // 32 for c in counts}
            assert nblk % world != 0 and len(words) > 1, (nblk, world, counts)
        assert sum(nx) > 0 and sum(nz) > 0
    elif name == "c1_ranks_without_candidates":
        assert min(nx) == 0 < max(nx), nx
    elif name == "c3_ranks_without_unsafe":
        assert min(nz) == 0 < max(nz), nz
    elif name == "c1_empty_safe_set":
        assert max(nx) == 0 and sum(nz) > 0, (nx, nz)


def _single_sets(engine, oracle, ds, lo, hi, grid, beta, rule, kernel, keep_v=0):
    """GPU posterior and sets of the unsharded context -> (P, mean, var, lcb, ucb, S, Z)."""
    capi = _capi()
    engine.set_grid(lo, hi, grid)
    engine.set_model(ds, kernel)
    m, v = engine.posterior(keep_v=keep_v)
    engine.sets(beta, _rule_id(rule))
    S, Z = engine.mask(capi.MASK_SAFE), engine.mask(capi.MASK_UNSAFE)
    lcb, ucb = oracle.bounds(m, v, beta)
    return oracle.make_grid(lo, hi, grid), m, v, lcb, ucb, S, Z


# ---------------------------------------------------------------------------------------------------------------------
# Lipschitz mode: SafeOpt expander split by candidates, GoOSE target on each rank's own z
# ---------------------------------------------------------------------------------------------------------------------
SO_KEYS = ("n_safe", "n_unsafe", "n_min", "min_ucb0", "min_ucb0_idx", "minimizer_idx", "minimizer_var", "expander_idx",
           "x_new_idx")
GO_KEYS = ("n_safe", "n_unsafe", "min_lcb0", "min_lcb0_idx", "target_idx", "target_lcb", "x_new_idx", "explore_idx")
PAIR_KEYS = ("per_idx", "per_value", "best_idx", "best_value", "n_hit", "n_x", "n_z", "pairs_algorithmic")


def _summary(st, keys, pair):
    """The global part of a step result (what every rank must return identically)."""
    out = {k: st[k] for k in keys}
    out["L"] = [float(x) for x in st["L"]] if "L" in st else None
    out["pairs"] = {k: v for k, v in st[pair].items() if k != "local"}
    return out


def _lipschitz_reference(engine, oracle, name):
    key = ("lipschitz", name)
    if key in _REF:
        return _REF[key]
    capi = _capi()
    ds, lo, hi, grid, beta, rule, kernel = _workload(oracle, name)
    P, m, v, lcb, ucb, S, Z = _single_sets(engine, oracle, ds, lo, hi, grid, beta, rule, kernel)
    G = ds["Y_norm"].shape[1]
    ref = {"S": S, "Z": Z, "mult": {}}
    Lg = None
    for mult in (1, 5):
        L = None if mult == 1 else np.full(G, mult * Lg[G - 1])
        st = engine.safeopt_step(ds, beta, unsafe_rule=_rule_id(rule), L=L, kernel=kernel)
        em = [engine.mask(capi.MASK_EXPANDER, c) for c in range(G - 1)]
        gs = engine.goose_step(ds, beta, unsafe_rule=_rule_id(rule), L=L, kernel=kernel)
        tm = [engine.mask(capi.MASK_TARGET, c) for c in range(G - 1)]
        if mult == 1:
            Lg = st["L"]
        Lo = np.full(G, mult * Lg[G - 1])
        ref["mult"][mult] = {"so": st, "go": gs, "em": em, "tm": tm, "L": L,
                             "exo": oracle.expander_lipschitz(P, S, Z, ucb, v, Lo)["masks"],
                             "tgo": oracle.goose_target(P, S, Z, ucb, lcb, Lo)["masks"]}
    if kernel != "RBF":        # the same data under the SE kernel: the kernel must change what the ranks compute
        engine.set_model(ds)
        engine.posterior(with_grad=True, fetch=False)
        ref["L_rbf"] = engine.lipschitz()
    _REF[key] = ref
    return ref


@pytest.mark.gpu
@pytest.mark.parametrize("name,world,block", LAYOUTS)
def test_lipschitz_ranks_match_one_context_and_the_oracle(engine, oracle, sharded, name, world, block):
    capi = _capi()
    ds, lo, hi, grid, beta, rule, kernel = _workload(oracle, name)
    ref = _lipschitz_reference(engine, oracle, name)
    G, N = ds["Y_norm"].shape[1], ref["S"].size
    nc = G - 1

    def body(eng, rank, g):
        infos = _record_prepare(eng)
        out = {"count": eng.count, "mult": {}}
        for mult, r in ref["mult"].items():
            st = sharded.safeopt_step(eng, ds, beta, unsafe_rule=_rule_id(rule), L=r["L"], group=g, kernel=kernel)
            so_info = infos[-1]
            em = [eng.mask(capi.MASK_EXPANDER, c) for c in range(nc)]
            sets = (eng.mask(capi.MASK_SAFE), eng.mask(capi.MASK_UNSAFE))
            gs = sharded.goose_step(eng, ds, beta, unsafe_rule=_rule_id(rule), L=r["L"], group=g, kernel=kernel)
            tm = [eng.mask(capi.MASK_TARGET, c) for c in range(nc)]
            out["mult"][mult] = {"so": _summary(st, SO_KEYS, "expander"), "go": _summary(gs, GO_KEYS, "target"),
                                 "em": em, "tm": tm, "sets": sets, "nx": int(so_info["n_x_local"]),
                                 "nz": int(so_info["n_z_local"])}
        return out

    res = run_ranks(world, _gpu_engines(lo, hi, grid, block), body)
    counts = [r["count"] for r in res]
    for mult, r in ref["mult"].items():
        loc = [x["mult"][mult] for x in res]
        if mult == 1:
            _assert_edge(name, world, block, N, counts, [x["nx"] for x in loc], [x["nz"] for x in loc])
        for x in loc[1:]:                                           # every rank returns the same global result
            assert x["so"] == loc[0]["so"] and x["go"] == loc[0]["go"], (mult, x["so"], loc[0]["so"])
        so, go = loc[0]["so"], loc[0]["go"]
        S = to_global([x["sets"][0] for x in loc], world, N, block)
        Z = to_global([x["sets"][1] for x in loc], world, N, block)
        assert np.array_equal(S, ref["S"]) and np.array_equal(Z, ref["Z"])
        assert [x["nx"] for x in loc] == [int(x["sets"][0].sum()) for x in loc]
        rso, rgo = r["so"], r["go"]
        if mult == 1:
            assert so["L"] == [float(x) for x in rso["L"]]             # all-reduce max of the ranks' Lipschitz constants
            if kernel != "RBF":
                assert so["L"][-1] != ref["L_rbf"][-1]
        for k in SO_KEYS:
            assert so[k] == rso[k], (mult, k, so[k], rso[k])
        for k in GO_KEYS:
            assert go[k] == rgo[k], (mult, k, go[k], rgo[k])
        for k in PAIR_KEYS:
            assert so["pairs"][k] == rso["expander"][k], (mult, "expander", k)
            assert go["pairs"][k] == rgo["target"][k], (mult, "target", k)
        a, b = rso["expander"]["pairs_evaluated"], so["pairs"]["pairs_evaluated"]
        assert b <= 1.1 * a + 4 * 256 * 256 * 3, (mult, a, b)
        for c in range(nc):
            em = to_global([x["em"][c] for x in loc], world, N, block)
            tm = to_global([x["tm"][c] for x in loc], world, N, block)
            assert np.array_equal(em, r["em"][c]), (mult, c, np.flatnonzero(em != r["em"][c])[:10])
            assert np.array_equal(tm, r["tm"][c]), (mult, c, np.flatnonzero(tm != r["tm"][c])[:10])
            assert (em != r["exo"][c]).sum() <= 2 and (tm != r["tgo"][c]).sum() <= 2     # threshold rounding only
        print(f"lipschitz {name} {world}x{block} L x{mult}: |S| {S.sum()} |Z| {Z.sum()} expander hits {so['pairs']['n_hit']} "
              f"target hits {go['pairs']['n_hit']}; pairs evaluated {b} (one context {a})")


# ---------------------------------------------------------------------------------------------------------------------
# fantasy mode: SafeOpt counts per candidate, GoOSE target over each rank's own z
# ---------------------------------------------------------------------------------------------------------------------
def _oracle_fantasy(oracle, P, ds, beta, S, Z, var, lcb, kernel):
    """FP64 counts (N,), target set (N,), and per pair the exact-rounding band: near_x (|S|,) pairs per candidate and
    near_z (N,) z with a pair within EXACT_TOL * sf2 * (1 + gain(x)) of the threshold."""
    if kernel == "RBF":
        counts = oracle.fantasy_counts(P, ds, beta, S, Z)
        T = goose_target_fantasy(P, ds, beta, S, Z, lcb)["mask"]
        margin = np.abs(oracle.fantasy_margin(P, ds, beta, S, Z))
    else:
        import matern_ref
        counts, T = matern_ref.fantasy_pairs(P, ds, beta, S, Z, kernel)
        margin = np.abs(matern_ref.fantasy_margin(P, ds, beta, S, Z, kernel))
    d, G = P.shape[1], ds["Y_norm"].shape[1]
    gain, sf2max = np.zeros(int(S.sum())), 0.0
    for i in range(1, G):
        _, sf2, sn2 = oracle.unpack_hyper(ds["hypopt"][:, i], d)
        sf2max = max(sf2max, sf2)
        vn = var[S, i] / ds["Y_std"][i] ** 2
        gain = np.maximum(gain, beta * np.sqrt(vn) / (vn + sn2 + oracle.EPS_F32))
    near = margin <= EXACT_TOL * sf2max * (1.0 + gain)[None, :]
    near_z = np.zeros(S.size, dtype=bool)
    near_z[np.flatnonzero(Z)] = near.any(axis=1)
    return np.asarray(counts, dtype=np.int64), np.asarray(T, dtype=bool), near.sum(axis=0), near_z


def _fantasy_reference(engine, oracle, name):
    key = ("fantasy", name)
    if key in _REF:
        return _REF[key]
    capi = _capi()
    ds, lo, hi, grid, beta, rule, kernel = _workload(oracle, name)
    P, m, v, lcb, ucb, S, Z = _single_sets(engine, oracle, ds, lo, hi, grid, beta, rule, kernel, keep_v=1)
    ref = {"S": S, "Z": Z, "so": {}, "go": {}}
    ref["counts_o"], ref["T_o"], ref["near_x"], ref["near_z"] = _oracle_fantasy(oracle, P, ds, beta, S, Z, v, lcb, kernel)
    for p in FANTASY_PRECISIONS:
        prec = capi.PRECISIONS[p][0]
        st = engine.safeopt_step(ds, beta, mode="fantasy", precision=p, unsafe_rule=_rule_id(rule), kernel=kernel)
        mask = engine.mask(capi.MASK_EXPANDER, 0)
        ex = engine.expander(beta, None, capi.MODE_FANTASY, prec, want_counts=True)
        ref["so"][p] = {"st": st, "mask": mask, "counts": ex["counts"].astype(np.int64)}
    for p in TARGET_PRECISIONS:
        gs = engine.goose_step(ds, beta, _rule_id(rule), mode="fantasy", precision=p, kernel=kernel)
        ref["go"][p] = {"st": gs, "T": engine.mask(capi.MASK_TARGET, 0)}
    _REF[key] = ref
    return ref


def _fantasy_rank_body(sharded, ds, beta, rule, kernel, precisions=FANTASY_PRECISIONS, targets=TARGET_PRECISIONS):
    capi = _capi()

    def body(eng, rank, g):
        infos = _record_prepare(eng)
        dev = torch.device("cuda", eng.device)
        out = {"count": eng.count, "so": {}, "go": {}}
        for p in precisions:
            prec, kv = capi.PRECISIONS[p]
            st = sharded.safeopt_step(eng, ds, beta, mode="fantasy", precision=p, unsafe_rule=_rule_id(rule), group=g,
                                      kernel=kernel)
            info = infos[-1]
            mask = eng.mask(capi.MASK_EXPANDER, 0)
            sharded._posterior_and_sets(eng, ds, beta, _rule_id(rule), with_grad=False, keep_v=kv, upload=False, device=dev,
                                        group=g, kernel=kernel)
            ex = sharded._pairs(eng, capi.MODE_FANTASY, prec, beta, None, False, dev, g, want_counts=True)
            out["so"][p] = {"sum": _summary(st, SO_KEYS, "expander"), "mask": mask, "counts": ex["local"]["counts"],
                            "n_hit": ex["n_hit"], "n_x": ex["n_x"], "nx": int(info["n_x_local"]), "nz": int(info["n_z_local"]),
                            "refine": eng.refine_stats(), "n_ambiguous_local": ex["local"]["n_ambiguous"]}
        for p in targets:
            gs = sharded.goose_step(eng, ds, beta, _rule_id(rule), mode="fantasy", precision=p, group=g, kernel=kernel)
            out["go"][p] = {"sum": _summary(gs, GO_KEYS, "target"), "T": eng.mask(capi.MASK_TARGET, 0)}
        return out
    return body


def _check_fantasy(ref, res, world, block, precisions=FANTASY_PRECISIONS, targets=TARGET_PRECISIONS, tag=""):
    N = ref["S"].size
    S = ref["S"]
    for p in precisions:
        loc = [x["so"][p] for x in res]
        for x in loc[1:]:
            assert x["sum"] == loc[0]["sum"], (p, x["sum"], loc[0]["sum"])
        got = to_global([x["counts"] for x in loc], world, N, block, np.int64)
        mask = to_global([x["mask"] for x in loc], world, N, block)
        one = ref["so"][p]
        assert not got[~S].any()
        near = ref["near_x"]
        # n_ambiguous depends on the shard (the error-bound maxima are taken over the local z): not compared
        for what, want in (("one context", one["counts"]), ("FP64 oracle", ref["counts_o"])):
            bad = np.flatnonzero(np.abs(got[S] - want[S]) > near)
            assert bad.size == 0, (tag, p, what, np.flatnonzero(S)[bad][:10], got[S][bad][:10], want[S][bad][:10])
        assert np.array_equal(mask, one["mask"]) and np.array_equal(mask, got > 0), p
        s, st = loc[0]["sum"], one["st"]
        assert s["pairs"]["n_hit"] == st["expander"]["n_hit"] == loc[0]["n_hit"] == int(mask.sum()), p
        assert s["pairs"]["n_x"] == st["expander"]["n_x"] == S.sum()
        for k in ("x_new_idx", "expander_idx", "minimizer_idx", "n_safe", "n_unsafe"):
            assert s[k] == st[k], (p, k, s[k], st[k])
        print(f"fantasy {tag} {world}x{block} {p}: n_x {S.sum()}, hits {int(mask.sum())}, newly safe {int(got.sum())}, "
              f"ambiguous per rank {[x['n_ambiguous_local'] for x in loc]}, refine {[x['refine'] for x in loc]}")
    for p in targets:
        loc = [x["go"][p] for x in res]
        for x in loc[1:]:
            assert x["sum"] == loc[0]["sum"], (p, x["sum"], loc[0]["sum"])
        T = to_global([x["T"] for x in loc], world, N, block)
        one = ref["go"][p]
        for what, want in (("one context", one["T"]), ("FP64 reference", ref["T_o"])):
            bad = np.flatnonzero((T != want) & ~ref["near_z"])
            assert bad.size == 0, (tag, p, what, bad[:10])
        s, st = loc[0]["sum"], one["st"]
        for k in ("target_idx", "x_new_idx", "explore_idx", "min_lcb0_idx"):
            assert s[k] == st[k], (p, k, s[k], st[k])
        assert s["pairs"]["n_hit"] == int(T.sum())


@pytest.mark.gpu
@pytest.mark.parametrize("name,world,block", LAYOUTS)
def test_fantasy_ranks_match_one_context_and_the_oracle(engine, oracle, sharded, name, world, block):
    ds, lo, hi, grid, beta, rule, kernel = _workload(oracle, name)
    ref = _fantasy_reference(engine, oracle, name)
    res = run_ranks(world, _gpu_engines(lo, hi, grid, block), _fantasy_rank_body(sharded, ds, beta, rule, kernel))
    loc = [x["so"]["fp64"] for x in res]
    _assert_edge(name, world, block, ref["S"].size, [x["count"] for x in res], [x["nx"] for x in loc], [x["nz"] for x in loc])
    if name == "c1_empty_safe_set":
        assert all(x["so"][p]["n_x"] == 0 for x in res for p in FANTASY_PRECISIONS)       # n_total = 0 in every precision
    _check_fantasy(ref, res, world, block, tag=name)


@pytest.mark.gpu
def test_refinement_cells_and_list_overflow_on_every_rank(engine, oracle, sharded):
    """npad = 256, three constraints, tf32: the FP64 refinement of each rank's ambiguous pairs (candidates of every rank
    against the rank's own z) cut into several cells by a small fantasy_refine_mb, and separately re-run after a list
    overflow (fantasy_refine_cap = 16).  Both give the counts of the default pass, which are those of one context."""
    ds, lo, hi, grid, beta, rule, kernel = _workload(oracle, "small_d4")
    world, block = 3, 64
    assert (ds["X_norm"].shape[0] + 63) // 64 * 64 == 256 and ds["Y_norm"].shape[1] == 4
    ref = _fantasy_reference(engine, oracle, "small_d4")
    body = _fantasy_rank_body(sharded, ds, beta, rule, kernel, precisions=("tf32",), targets=())
    runs = {}
    for label, opts in (("default", ()), ("cells", (("fantasy_refine_mb", 2),)), ("overflow", (("fantasy_refine_cap", 16),))):
        runs[label] = run_ranks(world, _gpu_engines(lo, hi, grid, block, opts), body)
        _check_fantasy(ref, runs[label], world, block, precisions=("tf32",), targets=(), tag=f"small d=4 {label}")
    for r in range(world):
        base, cut, ov = (runs[k][r]["so"]["tf32"] for k in ("default", "cells", "overflow"))
        assert base["refine"]["cells"] == 1 and base["n_ambiguous_local"] > 16, (r, base["refine"], base["n_ambiguous_local"])
        assert cut["refine"]["cells"] > 1, (r, cut["refine"])
        assert ov["n_ambiguous_local"] == base["n_ambiguous_local"] > 16
        assert np.array_equal(cut["counts"], base["counts"]) and np.array_equal(ov["counts"], base["counts"]), r


# ---------------------------------------------------------------------------------------------------------------------
# bounds mode (fantasy_refine = 3)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_goose_bounds_mode_on_three_ranks_brackets_the_fp64_target(engine, oracle, sharded):
    """The undecided unsafe points are local, so the torch path allows bounds mode for the GoOSE target: the certified set
    is inside the FP64 target set, which is inside certified + undecided."""
    capi = _capi()
    name, world, block = "c3_ragged", 3, 32
    ds, lo, hi, grid, beta, rule, kernel = _workload(oracle, name)
    ref = _fantasy_reference(engine, oracle, name)
    N, Tx, exact = ref["S"].size, ref["go"]["fp64"]["T"], ref["go"]["fp64"]["st"]

    def body(eng, rank, g):
        gs = sharded.goose_step(eng, ds, beta, _rule_id(rule), mode="fantasy", precision="tf32", group=g)
        return {"sum": _summary(gs, GO_KEYS, "target"), "T": eng.mask(capi.MASK_TARGET, 0), "refine": eng.refine_stats(),
                "und": {k: gs["target"][k] for k in ("n_undecided", "undecided_best_idx", "undecided_best_value")}}

    res = run_ranks(world, _gpu_engines(lo, hi, grid, block, (("fantasy_refine", 3),)), body)
    for x in res[1:]:
        assert x["sum"] == res[0]["sum"] and x["und"] == res[0]["und"]
    Tc = to_global([x["T"] for x in res], world, N, block)
    tg, und = res[0]["sum"]["pairs"], res[0]["und"]
    print(f"bounds {name} {world}x{block}: certified {tg['n_hit']}, undecided {und['n_undecided']}, FP64 {int(Tx.sum())}")
    assert all(x["refine"] == {"cells": 0, "fp64_rows": 0} for x in res)
    assert tg["n_hit"] == Tc.sum()
    assert not (Tc & ~Tx).any()
    assert Tx.sum() <= tg["n_hit"] + und["n_undecided"]
    if und["n_undecided"] == 0:
        assert np.array_equal(Tc, Tx)
    else:
        assert und["undecided_best_idx"] >= 0 and not Tc[und["undecided_best_idx"]]
    if und["undecided_best_value"] > tg["best_value"]:
        assert res[0]["sum"]["target_idx"] == exact["target_idx"]


@pytest.mark.gpu
def test_safeopt_bounds_mode_on_several_ranks_is_refused(engine, oracle, sharded):
    """The per-candidate undecided counts would need a combining all-reduce the torch path does not do."""
    name, world, block = "c3_ragged", 3, 32
    ds, lo, hi, grid, beta, rule, kernel = _workload(oracle, name)

    def body(eng, rank, g):
        with pytest.raises(ValueError, match="bounds mode"):
            sharded.safeopt_step(eng, ds, beta, mode="fantasy", precision="tf32", unsafe_rule=_rule_id(rule), group=g)
        return True

    assert run_ranks(world, _gpu_engines(lo, hi, grid, block, (("fantasy_refine", 3),)), body) == [True] * world
