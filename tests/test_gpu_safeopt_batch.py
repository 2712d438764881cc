"""GPU: the batch SafeOpt acquisition (csrc/batch.cu) against the NumPy reference (tests/safeopt_batch_ref.py), on one GPU,
sharded over thread ranks on one GPU and over the library's communicator on several GPUs."""
import numpy as np
import pytest
import torch      # before the library loads NCCL: torch links its own NCCL build

import safeopt_batch_ref as B
from conftest import golden_ds, load_golden
from test_gpu_sharded_ranks import THREAD_DIST, run_ranks

pytestmark = pytest.mark.gpu
RTOL = 1e-9
Q = 8
SMALL = [(3, 14, 70, 3, "all", 33), (4, 9, 200, 4, "any", 34), (6, 5, 130, 3, "any", 26)]   # (d, points per axis, n, G, rule, seed)
GOLD = [("c1_benoit", 9, 3.0, [48, 40], "all"), ("c3_wor", 20, 2.0, [45, 61], "any")]
MODES = [("lipschitz", "fp64"), ("fantasy", "fp64"), ("fantasy", "tf32")]


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


CASES = [f"small{i}" for i in range(len(SMALL))] + [g[0] for g in GOLD]


class _DeviceF64:
    def __init__(self, ptr, shape):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": "<f8", "data": (int(ptr), False), "strides": None,
                                         "version": 3}


def _state(eng):
    """Mean, var (read on the device, without recomputing them) and every mask the step left."""
    capi = _capi()
    out = {}
    for name, ptr in zip(("mean", "var"), eng.posterior_dev()):
        out[name] = torch.as_tensor(_DeviceF64(ptr, (eng.G, eng.count)), device="cuda:0").cpu().numpy().copy()
    for kind in (capi.MASK_SAFE, capi.MASK_MIN, capi.MASK_UNSAFE):
        out[f"mask{kind}"] = eng.mask(kind)
    for c in range(max(eng.G - 1, 1)):
        out[f"exp{c}"] = eng.mask(capi.MASK_EXPANDER, c)
    return out


def _step(eng, name, mode, prec, kernel):
    capi = _capi()
    ds, lo, hi, grid, beta, rule = _case(name)
    eng.set_grid(lo, hi, grid)
    st = eng.safeopt_step(ds, beta, mode=mode, precision=prec, kernel=kernel,
                          unsafe_rule=capi.UNSAFE_ANY if rule == "any" else capi.UNSAFE_ALL)
    return ds, lo, hi, grid, beta, rule, st


def _reference(eng, ds, lo, hi, grid, kernel, state, q, forced):
    from oracle import gp_oracle as O
    capi = _capi()
    E = np.zeros(eng.count, dtype=bool)
    for c in range(max(eng.G - 1, 1)):
        E |= state[f"exp{c}"]
    return B.safeopt_batch(O.make_grid(lo, hi, grid), ds, state["var"][0], state[f"mask{capi.MASK_MIN}"], E, q, kernel=kernel,
                           forced=forced, rtol=RTOL)


def _compare(got, ref, tag):
    """Picks equal the reference's, stds to RTOL; a pick decided inside RTOL is reported and skipped."""
    assert len(got) == len(ref), tag
    skipped = 0
    for b, (g, r) in enumerate(zip(got, ref)):
        for k in ("std_min", "std_exp"):
            assert g[k] == pytest.approx(r[k], rel=RTOL, abs=1e-300), (tag, b, k)
        if r["near_tie"]:
            skipped += 1
            print(f"{tag}: pick {b} decided within {RTOL} of a tie (gpu {g['idx']}, reference {r['idx']}): skipped")
            continue
        assert (g["idx"], g["from_expander"], g["idx_min"], g["idx_exp"]) == (r["idx"], r["from_expander"], r["idx_min"], r["idx_exp"]), (tag, b)
    assert skipped < len(got) or not got, tag
    return skipped


@pytest.mark.parametrize("kernel", ["RBF", "Matern52"])
@pytest.mark.parametrize("mode,prec", MODES)
@pytest.mark.parametrize("name", CASES)
def test_batch_matches_the_reference_and_leaves_the_step_alone(engine, name, mode, prec, kernel):
    ds, lo, hi, grid, beta, rule, st = _step(engine, name, mode, prec, kernel)
    before = _state(engine)
    engine.kernel_launches(reset=True)
    picks = engine.safeopt_batch(Q)
    launches = engine.kernel_launches()
    after = _state(engine)
    for k in before:
        assert np.array_equal(before[k], after[k]), k
    assert launches <= 3 * Q + 8, launches
    if st["minimizer_idx"] < 0 and st["expander_idx"] < 0:     # M and E empty: no pick
        assert picks == [] and _reference(engine, ds, lo, hi, grid, kernel, before, Q, None) == []
        return
    assert len(picks) == Q
    x_new = st["x_new_idx"] if st["x_new_idx"] >= 0 else st["minimizer_idx"]
    assert picks[0]["idx"] == x_new
    assert picks[0]["std_min"] == st["minimizer_std"] and picks[0]["std_exp"] == st["expander_std"]
    ref = _reference(engine, ds, lo, hi, grid, kernel, before, Q, [p["idx"] for p in picks])
    _compare(picks, ref, f"{name} {mode} {prec} {kernel}")
    assert engine.safeopt_batch(1)[0] == picks[0]          # q = 1: the step's x_new; the batch can be repeated


def test_errors(engine):
    capi = _capi()
    ds, lo, hi, grid, beta, rule = _case("small0")
    engine.set_grid(lo, hi, grid)
    with pytest.raises(ValueError, match="SafeOpt pair stage"):
        engine.safeopt_batch(4)                             # no step since the grid was set
    engine.safeopt_step(ds, beta)
    for q in (0, -1, capi.BATCH_MAX_Q + 1):
        with pytest.raises(ValueError, match="out of range"):
            engine.safeopt_batch(q)
    assert len(engine.safeopt_batch(capi.BATCH_MAX_Q)) == capi.BATCH_MAX_Q
    engine.set_model(ds)
    with pytest.raises(ValueError, match="SafeOpt pair stage"):
        engine.safeopt_batch(4)
    engine.safeopt_step(ds, beta)
    engine.goose_step(ds, beta)
    with pytest.raises(ValueError, match="SafeOpt pair stage"):
        engine.safeopt_batch(4)
    engine.safeopt_step(ds, beta)
    engine.batch_prepare(2)
    engine.batch_local()
    engine.posterior(fetch=False)
    with pytest.raises(ValueError, match="no prepared batch"):
        engine.batch_local()
    engine.safeopt_step(ds, beta)
    engine.batch_prepare(1)
    engine.batch_commit(engine.batch_local()["idx"])
    with pytest.raises(ValueError, match="committed"):
        engine.batch_local()


def test_explicit_points_give_the_meshgrid_picks(engine):
    """sbo_set_points: every pick's coordinates come from its global index on the explicit points too."""
    from oracle import gp_oracle as O
    ds, lo, hi, grid, beta, rule, st = _step(engine, "small1", "lipschitz", "fp64", "RBF")
    mesh = engine.safeopt_batch(Q)
    engine.set_points(O.make_grid(lo, hi, grid))
    engine.safeopt_step(ds, beta, unsafe_rule=_capi().UNSAFE_ANY)
    pts = engine.safeopt_batch(Q)
    assert [p["idx"] for p in pts] == [p["idx"] for p in mesh]
    for a, b in zip(pts, mesh):
        assert a["std_exp"] == pytest.approx(b["std_exp"], rel=1e-12) and a["std_min"] == pytest.approx(b["std_min"], rel=1e-12)


def test_c4_full_size_q16(engine):
    from sbo_b200 import workloads
    capi = _capi()
    ds, lo, hi, grid, beta = workloads.c4()
    engine.set_grid(lo, hi, grid)
    st = engine.safeopt_step(ds, beta, mode="fantasy", precision="tf32", unsafe_rule=capi.UNSAFE_ANY)
    state = _state(engine)
    picks = engine.safeopt_batch(16)
    assert picks[0]["idx"] == st["x_new_idx"]
    ref = _reference(engine, ds, lo, hi, grid, "RBF", state, 16, [p["idx"] for p in picks])
    _compare(picks, ref, "C4")
    n_cand = int((state[f"mask{capi.MASK_MIN}"] | state["exp0"]).sum())
    assert 0 < n_cand <= st["n_safe"]


@pytest.fixture
def sharded(monkeypatch):
    import sbo_b200  # noqa: F401
    from sbo_b200 import sharded as mod
    monkeypatch.setattr(mod, "dist", THREAD_DIST)
    return mod


@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("name,mode,prec,kernel", [("c3_wor", "lipschitz", "fp64", "RBF"), ("small1", "fantasy", "fp64", "Matern52")])
def test_thread_ranks_give_the_unsharded_picks(engine, sharded, world, name, mode, prec, kernel):
    import sbo_b200
    capi = _capi()
    ds, lo, hi, grid, beta, rule, _ = _step(engine, name, mode, prec, kernel)
    single = engine.safeopt_batch(Q)
    rid = capi.UNSAFE_ANY if rule == "any" else capi.UNSAFE_ALL
    N = int(np.prod(grid))

    def make(rank, w):
        eng = sbo_b200.GridEngine(0)
        eng.set_grid(lo, hi, grid)
        eng.set_shard_cyclic(rank, w, 32)
        return eng

    def body(eng, rank, g):
        sharded.safeopt_step(eng, ds, beta, mode=mode, precision=prec, unsafe_rule=rid, group=g, kernel=kernel)
        return sharded.safeopt_batch(eng, Q, device=torch.device("cuda", 0), group=g), eng.count

    res = run_ranks(world, make, body)
    assert sum(c for _, c in res) == N
    for picks, _ in res:
        assert picks == res[0][0]
    got = res[0][0]
    assert [p["idx"] for p in got] == [p["idx"] for p in single]
    for a, b in zip(got, single):
        assert a["from_expander"] == b["from_expander"] and (a["idx_min"], a["idx_exp"]) == (b["idx_min"], b["idx_exp"])
        assert a["std_min"] == pytest.approx(b["std_min"], rel=1e-12) and a["std_exp"] == pytest.approx(b["std_exp"], rel=1e-12)


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
eng.safeopt_step_sharded(ds, beta, unsafe_rule=1)
got = [p["idx"] for p in eng.safeopt_batch_sharded(8)]
if rank == 0:
    one = sbo_b200.GridEngine(0)
    one.set_grid(lo, hi, pts)
    one.safeopt_step(ds, beta, unsafe_rule=1)
    ref = [p["idx"] for p in one.safeopt_batch(8)]
    assert got == ref, (got, ref)
    print("ok", got)
eng.close()
dist.destroy_process_group()
"""
    env = dict(os.environ, SBO_ROOT=ROOT, MASTER_ADDR="127.0.0.1", MASTER_PORT="29533", WORLD_SIZE="2")
    procs = [subprocess.Popen([sys.executable, "-c", code], env=dict(env, RANK=str(r)), stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                              text=True) for r in range(2)]
    outs = [p.communicate(timeout=600)[0] for p in procs]
    assert all(p.returncode == 0 for p in procs), outs
    assert "ok" in outs[0]
