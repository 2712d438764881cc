"""GPU: what a change to the context leaves valid of a staged pair stage and a prepared batch (stage_changed, csrc/capi.cu).

A model, sample, grid, point-set, shard, posterior or sets-pass-1 change makes a prepared pair stage stale: each of its
remaining staged calls fails with ValueError and launches nothing.  sbo_release(1) stops a prepared fantasy stage from
exporting the V rows it frees, while a stage that has exported imports, runs and finishes to the same result.
sbo_release(2) after the finish leaves the expander mask and a prepared batch usable, and a new pair stage or finish drops a
prepared batch.  Every change keeps the number of grid points, so a stale stage's indices would still fit its masks."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

D, PPD, N0, G, SEED = 3, 12, 40, 3, 7
CHANGES = ["set_model", "set_model_ex", "append_sample", "posterior_update", "set_grid", "set_points", "set_shard",
           "set_shard_cyclic", "posterior", "sets_pass1"]


def _capi():
    from sbo_b200 import _capi
    return _capi


@pytest.fixture(scope="module")
def eng():
    import sbo_b200
    e = sbo_b200.GridEngine(0)
    yield e
    e.close()


@pytest.fixture(scope="module")
def case():
    """(ds0, ds1, lo, hi, pts, beta): N0 installed samples, and the same data set with one more (same normalisation)."""
    from sbo_b200 import workloads
    ds1, lo, hi, pts, beta = workloads.small(d=D, pts_per_dim=PPD, n=N0 + 1, seed=SEED, G=G)
    ds0 = dict(ds1, X_norm=ds1["X_norm"][:N0], Y_norm=ds1["Y_norm"][:N0])
    return ds0, ds1, lo, hi, pts, beta


def _start(eng, case, mode, precision="fp64"):
    """Grid, model, posterior, both sets passes and sbo_pairs_prepare; the stage's device buffers."""
    capi = _capi()
    ds0, _, lo, hi, pts, beta = case
    fantasy = mode == "fantasy"
    prec, kv = capi.PRECISIONS[precision]
    eng.set_grid(lo, hi, pts)
    eng.set_model(ds0)
    eng.posterior(with_grad=not fantasy, keep_v=kv if fantasy else 0, fetch=False)
    eng.sets(beta, capi.UNSAFE_ANY)
    L = None if fantasy else np.full(G, eng.lipschitz()[G - 1])
    info = eng.pairs_prepare(capi.MODE_FANTASY if fantasy else capi.MODE_LIPSCHITZ, prec, beta, L)
    nx = info["n_x_local"]
    assert nx > 0 and info["n_z_local"] > 0, "the case must pair something"
    st = {"fantasy": fantasy, "nx": nx,
          "rows": torch.zeros((nx, info["row_doubles"]), dtype=torch.float64, device="cuda"),
          "vrows": torch.zeros((nx, info["vrow_bytes"]), dtype=torch.uint8, device="cuda") if fantasy else None,
          "result": torch.zeros(4 * nx if fantasy else (G - 1) * nx, dtype=torch.uint8, device="cuda")}
    torch.cuda.synchronize()              # the library works on its own stream
    return st


def _calls(eng, st):
    return {"export": lambda: eng.pairs_export(st["rows"], st["vrows"]),
            "import": lambda: eng.pairs_import(st["nx"], st["rows"], st["vrows"]),
            "run": lambda: eng.pairs_run(False, st["result"]),
            "finish": lambda: eng.pairs_finish(False, 0, st["result"], want_counts=st["fantasy"])}


def _complete(eng, st, release_after_export=False):
    calls = _calls(eng, st)
    calls["export"]()
    if release_after_export:
        eng.release(1)
    calls["import"]()
    calls["run"]()
    return calls["finish"]()


def _change(eng, case, mode, name):
    from oracle import gp_oracle as O
    capi = _capi()
    ds0, ds1, lo, hi, pts, beta = case
    fantasy = mode == "fantasy"
    if name in ("append_sample", "posterior_update"):
        eng.append_sample(ds1["X_norm"][N0], ds1["Y_norm"][N0])
        if name == "posterior_update":
            _, info = eng.posterior_update(fetch=False)
            assert info == {"rows": 1, "recomputed": False}
        return
    {"set_model": lambda: eng.set_model(ds0),
     "set_model_ex": lambda: eng.set_model(ds0, "Matern52"),
     "set_grid": lambda: eng.set_grid(lo, hi, pts),
     "set_points": lambda: eng.set_points(O.make_grid(lo, hi, pts)),
     "set_shard": lambda: eng.set_shard(0, eng.N),
     "set_shard_cyclic": lambda: eng.set_shard_cyclic(0, 1, 64),
     "posterior": lambda: eng.posterior(with_grad=not fantasy, keep_v=1 if fantasy else 0, fetch=False),
     "sets_pass1": lambda: eng.sets_pass1(beta, capi.UNSAFE_ANY)}[name]()


@pytest.mark.parametrize("change", CHANGES)
@pytest.mark.parametrize("after", ["prepare", "run"])
@pytest.mark.parametrize("mode", ["fantasy", "lipschitz"])
def test_a_change_makes_the_stage_stale(eng, case, mode, after, change):
    st = _start(eng, case, mode)
    calls = _calls(eng, st)
    left = ["export", "import", "run", "finish"]
    if after == "run":
        for name in left[:3]:
            calls[name]()
        left = left[2:]
    count = eng.count
    _change(eng, case, mode, change)
    assert eng.count == count
    for name in left:
        l0 = eng.kernel_launches()
        with pytest.raises(ValueError):
            calls[name]()
        assert eng.kernel_launches() == l0, name


def test_release_v_before_export_refuses_the_export(eng, case):
    st = _start(eng, case, "fantasy")
    eng.release(1)
    l0 = eng.kernel_launches()
    with pytest.raises(ValueError, match="sbo_pairs_export"):
        _calls(eng, st)["export"]()
    assert eng.kernel_launches() == l0


@pytest.mark.parametrize("precision", ["fp64", "tf32"])
def test_release_v_after_export_gives_the_same_result(eng, case, precision):
    capi = _capi()
    keys = ("best_idx", "best_value", "per_idx", "per_value", "n_x", "n_z", "n_hit")
    got = []
    for release in (False, True):
        st = _start(eng, case, "fantasy", precision)
        r = _complete(eng, st, release_after_export=release)
        got.append(({k: r[k] for k in keys}, r["counts"], eng.mask(capi.MASK_EXPANDER, 0)))
    (ra, ca, ma), (rb, cb, mb) = got
    assert ra == rb and np.array_equal(ca, cb) and np.array_equal(ma, mb)
    assert ra["n_hit"] > 0


def test_release_pairs_after_finish_keeps_the_masks_and_the_batch(eng, case):
    capi = _capi()
    _complete(eng, _start(eng, case, "fantasy"))
    exp = eng.mask(capi.MASK_EXPANDER, 0)
    picks = eng.safeopt_batch(4)
    assert len(picks) == 4
    eng.batch_prepare(2)
    eng.release(2)
    assert np.array_equal(eng.mask(capi.MASK_EXPANDER, 0), exp)
    assert eng.batch_local() == picks[0]
    assert eng.safeopt_batch(4) == picks


def test_a_new_pair_stage_or_finish_drops_a_prepared_batch(eng, case):
    capi = _capi()
    beta = case[-1]
    st = _start(eng, case, "fantasy")
    _complete(eng, st)
    for again in ("finish", "prepare"):
        eng.batch_prepare(2)
        idx = eng.batch_local()["idx"]
        if again == "finish":
            _calls(eng, st)["finish"]()
        else:
            eng.pairs_prepare(capi.MODE_FANTASY, capi.PREC_FP64, beta)
        l0 = eng.kernel_launches()
        with pytest.raises(ValueError, match="no prepared batch"):
            eng.batch_local()
        with pytest.raises(ValueError, match="no prepared batch"):
            eng.batch_commit(idx)
        assert eng.kernel_launches() == l0, again
