"""GPU: the batch GoOSE acquisition (csrc/batch.cu) against the NumPy reference (tests/goose_batch_ref.py), on one GPU,
sharded over thread ranks on one GPU and over the library's communicator on several GPUs."""
import numpy as np
import pytest
import torch      # before the library loads NCCL: torch links its own NCCL build

import goose_batch_ref as GB
from conftest import golden_ds, load_golden
from test_gpu_sharded_ranks import THREAD_DIST, run_ranks

pytestmark = pytest.mark.gpu
RTOL = 1e-9
Q = 8
SMALL = [(3, 14, 70, 3, "all", 33), (4, 9, 200, 4, "any", 34), (6, 5, 130, 3, "any", 26)]   # (d, points per axis, n, G, rule, seed)
GOLD = [("c1_benoit", 9, 3.0, [48, 40], "all"), ("c3_wor", 20, 2.0, [45, 61], "any")]
MODES = [("lipschitz", "fp64"), ("fantasy", "fp64"), ("fantasy", "tf32")]
CASES = [f"small{i}" for i in range(len(SMALL))] + [g[0] for g in GOLD]


def _capi():
    from sbo_b200 import _capi
    return _capi


def _case(name):
    from sbo_b200 import workloads
    if name.startswith("small"):
        d, ppd, n, G, rule, seed = SMALL[int(name[-1])]
        ds, lo, hi, pts, beta = workloads.small(d=d, pts_per_dim=ppd, n=n, seed=seed, G=G)
        return dict(ds), lo, hi, pts, beta, rule
    from oracle import gp_oracle as O
    gname, n, beta, grid, rule = next(g for g in GOLD if g[0] == name)
    gold = load_golden(gname)
    return golden_ds(O, gold, n), gold["lo"], gold["hi"], grid, beta, rule


class _DeviceF64:
    def __init__(self, ptr, shape):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": "<f8", "data": (int(ptr), False), "strides": None,
                                         "version": 3}


def _state(eng):
    """Mean, var (read on the device, without recomputing them), S, Z and the target masks the step left."""
    capi = _capi()
    out = {}
    for name, ptr in zip(("mean", "var"), eng.posterior_dev()):
        out[name] = torch.as_tensor(_DeviceF64(ptr, (eng.G, eng.count)), device="cuda:0").cpu().numpy().copy()
    out["S"] = eng.mask(capi.MASK_SAFE)
    out["Z"] = eng.mask(capi.MASK_UNSAFE)
    for c in range(max(eng.G - 1, 1)):
        out[f"tgt{c}"] = eng.mask(capi.MASK_TARGET, c)
    return out


def _target_union(state):
    T = np.zeros_like(state["S"])
    for k in state:
        if k.startswith("tgt"):
            T |= state[k]
    return T


def _step(eng, name, mode, prec, kernel):
    capi = _capi()
    ds, lo, hi, grid, beta, rule = _case(name)
    eng.set_grid(lo, hi, grid)
    st = eng.goose_step(ds, beta, mode=mode, precision=prec, kernel=kernel,
                        unsafe_rule=capi.UNSAFE_ANY if rule == "any" else capi.UNSAFE_ALL)
    return ds, lo, hi, grid, beta, rule, st


def _forced(picks):
    return [(p["idx"], p["target_idx"] if p["explore"] else -1) for p in picks]


def _reference(ds, lo, hi, grid, beta, kernel, state, q, forced):
    from oracle import gp_oracle as O
    return GB.goose_batch(O.make_grid(lo, hi, grid), ds, state["mean"][0], state["var"][0], beta, state["S"], _target_union(state), q,
                          kernel=kernel, forced=forced, rtol=RTOL)


def _compare(got, ref, tag):
    """Picks equal the reference's, lcbs to RTOL (of the largest |lcb_0| among them); a pick decided inside RTOL is reported
    and skipped."""
    assert len(got) == len(ref), tag
    vals = [abs(r[k]) for r in ref for k in ("safe_lcb", "target_lcb") if np.isfinite(r[k])]
    tol = RTOL * max(vals + [1e-300])
    skipped = 0
    for b, (g, r) in enumerate(zip(got, ref)):
        for k in ("safe_lcb", "target_lcb"):
            assert g[k] == pytest.approx(r[k], rel=RTOL, abs=tol), (tag, b, k)
        if r["near_tie"]:
            skipped += 1
            print(f"{tag}: pick {b} decided within {RTOL} of a tie (gpu {g['idx']}, reference {r['idx']}): skipped")
            continue
        assert (g["idx"], g["explore"], g["safe_idx"], g["target_idx"]) == (r["idx"], r["explore"], r["safe_idx"], r["target_idx"]), (tag, b)
        assert g["dist"] == pytest.approx(r["dist"], rel=1e-12, abs=1e-300), (tag, b)
    assert skipped < len(got) or not got, tag
    return skipped


def _check_pick_one(picks, st):
    p = picks[0]
    assert p["idx"] == st["x_new_idx"]
    assert (p["idx"] if p["explore"] else -1) == st["explore_idx"]
    assert p["safe_lcb"] == st["min_lcb0"] and p["target_lcb"] == st["target_lcb"]


@pytest.mark.parametrize("kernel", ["RBF", "Matern52"])
@pytest.mark.parametrize("mode,prec", MODES)
@pytest.mark.parametrize("name", CASES)
def test_batch_matches_the_reference_and_leaves_the_step_alone(engine, name, mode, prec, kernel):
    ds, lo, hi, grid, beta, rule, st = _step(engine, name, mode, prec, kernel)
    before = _state(engine)
    engine.kernel_launches(reset=True)
    picks = engine.goose_batch(Q)
    launches = engine.kernel_launches()
    after = _state(engine)
    for k in before:
        assert np.array_equal(before[k], after[k]), k
    assert launches <= 5 * Q + 8, launches
    n_safe = int(before["S"].sum())
    assert len(picks) == min(Q, n_safe)
    if n_safe == 0:                                            # S empty: no pick
        assert picks == [] and st["x_new_idx"] < 0
        assert _reference(ds, lo, hi, grid, beta, kernel, before, Q, None) == []
        return
    _check_pick_one(picks, st)
    assert len({p["idx"] for p in picks}) == len(picks) and all(before["S"][p["idx"]] for p in picks)
    ref = _reference(ds, lo, hi, grid, beta, kernel, before, Q, _forced(picks))
    _compare(picks, ref, f"{name} {mode} {prec} {kernel}")
    print(f"{name} {mode} {prec} {kernel}:", "".join("E" if p["explore"] else "S" for p in picks))
    assert engine.goose_batch(1)[0] == picks[0]                # q = 1: the step's x_new; the batch can be repeated


def test_both_branches_occur(engine):
    """c1_benoit (Lipschitz, RBF) explores at pick 1 and takes safe minima after it; small0 explores."""
    _step(engine, "c1_benoit", "lipschitz", "fp64", "RBF")
    picks = engine.goose_batch(Q)
    assert picks[0]["explore"] == 1 and any(p["explore"] == 0 for p in picks[1:])
    _step(engine, "small0", "lipschitz", "fp64", "RBF")
    assert engine.goose_batch(Q)[0]["explore"] == 1


def test_bounds_mode_uses_the_certified_target(engine):
    capi = _capi()
    for name in ("small1", "c3_wor"):
        engine.set_option("fantasy_refine", 3)
        try:
            ds, lo, hi, grid, beta, rule, st = _step(engine, name, "fantasy", "tf32", "RBF")
            state = _state(engine)
            picks = engine.goose_batch(Q)
            n_cand = engine.goose_batch_prepare(1)
        finally:
            engine.set_option("fantasy_refine", 2)
        T = _target_union(state)
        assert st["target"]["n_hit"] == T.sum() and n_cand == int((state["S"] | T).sum())
        _check_pick_one(picks, st)
        _compare(picks, _reference(ds, lo, hi, grid, beta, "RBF", state, Q, _forced(picks)), f"bounds {name}")
        assert capi.MASK_TARGET == 5


def test_errors(engine):
    capi = _capi()
    ds, lo, hi, grid, beta, rule = _case("small0")
    engine.set_grid(lo, hi, grid)
    with pytest.raises(ValueError, match="GoOSE target stage"):
        engine.goose_batch(4)                                  # no step since the grid was set
    st = engine.goose_step(ds, beta)
    for q in (0, -1, capi.BATCH_MAX_Q + 1):
        with pytest.raises(ValueError, match="out of range"):
            engine.goose_batch(q)
    assert len(engine.goose_batch(capi.BATCH_MAX_Q)) == min(capi.BATCH_MAX_Q, st["n_safe"])
    engine.set_model(ds)
    with pytest.raises(ValueError, match="GoOSE target stage"):
        engine.goose_batch(4)
    engine.goose_step(ds, beta)
    engine.safeopt_step(ds, beta)
    with pytest.raises(ValueError, match="GoOSE target stage"):
        engine.goose_batch(4)                                  # after a SafeOpt step
    engine.goose_step(ds, beta)
    first = engine.goose_batch(1)[0]
    engine.goose_batch_prepare(1)
    with pytest.raises(ValueError, match="no prepared batch"):
        engine.batch_local()                                   # the SafeOpt staged calls refuse a GoOSE batch
    p = engine.goose_batch_local()                             # one rank: the local optima are the global ones
    assert p["explore"] == first["explore"] and (p["idx"] == -1 if p["explore"] else p["idx"] == first["idx"])
    idx = engine.goose_batch_nearest(p["target_idx"])[0] if p["explore"] else p["idx"]   # an explore pick's point
    assert idx == first["idx"]
    engine.goose_batch_commit(idx, p["target_idx"] if p["explore"] else -1)
    with pytest.raises(ValueError, match="committed"):
        engine.goose_batch_commit(idx, -1)                     # commit past q
    with pytest.raises(ValueError, match="committed"):
        engine.goose_batch_local()
    engine.goose_batch_prepare(2)
    engine.posterior(fetch=False)
    with pytest.raises(ValueError, match="no prepared GoOSE batch"):
        engine.goose_batch_local()
    # a GoOSE batch leaves the SafeOpt batch of a later SafeOpt step alone
    engine.goose_step(ds, beta)
    engine.goose_batch(4)
    engine.safeopt_step(ds, beta)
    assert len(engine.safeopt_batch(4)) == 4


def test_explicit_points_give_the_meshgrid_picks(engine):
    """sbo_set_points: every pick's coordinates and distances come from its global index on the explicit points too."""
    from oracle import gp_oracle as O
    ds, lo, hi, grid, beta, rule, st = _step(engine, "small1", "lipschitz", "fp64", "RBF")
    mesh = engine.goose_batch(Q)
    engine.set_points(O.make_grid(lo, hi, grid))
    engine.goose_step(ds, beta, unsafe_rule=_capi().UNSAFE_ANY)
    pts = engine.goose_batch(Q)
    assert [(p["idx"], p["explore"], p["target_idx"]) for p in pts] == [(p["idx"], p["explore"], p["target_idx"]) for p in mesh]
    for a, b in zip(pts, mesh):
        assert a["safe_lcb"] == pytest.approx(b["safe_lcb"], rel=1e-12) and a["target_lcb"] == pytest.approx(b["target_lcb"], rel=1e-12)
        assert a["dist"] == pytest.approx(b["dist"], rel=1e-12)


def test_c4_full_size_q16(engine):
    from sbo_b200 import workloads
    capi = _capi()
    ds, lo, hi, grid, beta = workloads.c4()
    engine.set_grid(lo, hi, grid)
    st = engine.goose_step(ds, beta, mode="fantasy", precision="tf32", unsafe_rule=capi.UNSAFE_ANY)
    state = _state(engine)
    picks = engine.goose_batch(16)
    assert len(picks) == 16
    _check_pick_one(picks, st)
    ref = _reference(ds, lo, hi, grid, beta, "RBF", state, 16, _forced(picks))
    _compare(picks, ref, "C4")
    print("C4:", "".join("E" if p["explore"] else "S" for p in picks), "|C| =", int((state["S"] | _target_union(state)).sum()))


@pytest.fixture
def sharded(monkeypatch):
    import sbo_b200  # noqa: F401
    from sbo_b200 import sharded as mod
    monkeypatch.setattr(mod, "dist", THREAD_DIST)
    return mod


@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("name,mode,prec,kernel", [("c3_wor", "lipschitz", "fp64", "RBF"), ("c1_benoit", "lipschitz", "fp64", "RBF"),
                                                   ("small1", "fantasy", "fp64", "Matern52")])
def test_thread_ranks_give_the_unsharded_picks(engine, sharded, world, name, mode, prec, kernel):
    import sbo_b200
    capi = _capi()
    ds, lo, hi, grid, beta, rule, _ = _step(engine, name, mode, prec, kernel)
    single = engine.goose_batch(Q)
    rid = capi.UNSAFE_ANY if rule == "any" else capi.UNSAFE_ALL
    N = int(np.prod(grid))

    def make(rank, w):
        eng = sbo_b200.GridEngine(0)
        eng.set_grid(lo, hi, grid)
        eng.set_shard_cyclic(rank, w, 32)
        return eng

    def body(eng, rank, g):
        sharded.goose_step(eng, ds, beta, mode=mode, precision=prec, unsafe_rule=rid, group=g, kernel=kernel)
        return sharded.goose_batch(eng, Q, device=torch.device("cuda", 0), group=g), eng.count

    res = run_ranks(world, make, body)
    assert sum(c for _, c in res) == N
    for picks, _ in res:
        assert picks == res[0][0]
    got = res[0][0]
    assert [(p["idx"], p["explore"], p["safe_idx"], p["target_idx"]) for p in got] == \
        [(p["idx"], p["explore"], p["safe_idx"], p["target_idx"]) for p in single]
    for a, b in zip(got, single):
        assert a["safe_lcb"] == pytest.approx(b["safe_lcb"], rel=1e-12) and a["target_lcb"] == pytest.approx(b["target_lcb"], rel=1e-12)
        assert a["dist"] == pytest.approx(b["dist"], rel=1e-12)


def test_library_communicator_batch_on_several_gpus():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    import os
    import subprocess
    import sys
    from conftest import ROOT
    code = r"""
import os, sys, numpy as np, torch, torch.distributed as dist
sys.path.insert(0, os.environ["SBO_ROOT"])
import sbo_b200
from sbo_b200 import sharded, workloads
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(rank)
dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
ds, lo, hi, pts, beta = workloads.small(d=4, pts_per_dim=9, n=200, seed=34, G=4)
eng = sbo_b200.GridEngine(rank)
eng.set_grid(lo, hi, pts)
eng.set_shard_cyclic(rank, world, 32)
sharded.init_comm(eng)
eng.goose_step_sharded(ds, beta, unsafe_rule=1)
got = [(p["idx"], p["explore"]) for p in eng.goose_batch_sharded(8)]
if rank == 0:
    one = sbo_b200.GridEngine(0)
    one.set_grid(lo, hi, pts)
    one.goose_step(ds, beta, unsafe_rule=1)
    ref = [(p["idx"], p["explore"]) for p in one.goose_batch(8)]
    assert got == ref, (got, ref)
    print("ok", got)
eng.close()
dist.destroy_process_group()
"""
    env = dict(os.environ, SBO_ROOT=ROOT, MASTER_ADDR="127.0.0.1", MASTER_PORT="29534", WORLD_SIZE="2")
    procs = [subprocess.Popen([sys.executable, "-c", code], env=dict(env, RANK=str(r)), stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                              text=True) for r in range(2)]
    outs = [p.communicate(timeout=600)[0] for p in procs]
    assert all(p.returncode == 0 for p in procs), outs
    assert "ok" in outs[0]
