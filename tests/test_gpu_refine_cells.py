"""GPU: the FP64 refinement of the tensor-core fantasy expander cut into cells (option fantasy_refine_mb, csrc/pairs.cu
refine_ambiguous).  A pass whose FP64 rows do not fit its memory budget runs block of candidates by block of unsafe points;
every pair is still re-evaluated by the same FP64 arithmetic on the same FP64 rows, so the counts must be IDENTICAL to the
one-cell pass, and within the usual rounding tolerance of the FP64 kernel."""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu
GOLD = os.path.join(ROOT, "tests", "golden")
SMALL = [(4, 9, 200, 4, "any"), (3, 14, 70, 3, "all"), (6, 5, 130, 3, "any")]    # (d, points per axis, n, G, unsafe rule)


def _capi():
    from sbo_b200 import _capi
    return _capi


def _budget_mb(eng, ex, stats, frac):
    """A budget in MB whose FP64 rows hold about `frac` of the one-cell pass's rows: rows (constraints) and posterior
    scratch (all GPs) of npad doubles per point, the bucketed list, and the scratch floor of one 128-point chunk."""
    npad = (eng.n + 63) // 64 * 64
    per_point = (eng.G - 1 + eng.G) * npad * 8
    need = stats["fp64_rows"] * frac * per_point + ex["n_ambiguous"] * 8 + eng.G * npad * 128 * 8
    return max(1, int(np.ceil(need / 2 ** 20)))


def _forced(eng, run, ex, stats, min_cells, frac=1 / 6):
    """Run with a budget that cuts the pass into at least `min_cells` cells (lowered step by step until it does, or until
    the next lower budget is refused)."""
    from sbo_b200.engine import SboError
    mb, best = _budget_mb(eng, ex, stats, frac), None
    try:
        while mb >= 1:
            eng.set_option("fantasy_refine_mb", mb)
            try:
                r = run()
            except SboError:
                if best is None:
                    raise
                break
            best = (mb, r, eng.refine_stats())
            if best[2]["cells"] >= min_cells:
                break
            mb = min(mb - 1, mb * 3 // 4)
    finally:
        eng.set_option("fantasy_refine_mb", 0)
    return best


def _small(engine, d, ppd, n, G, rule):
    capi = _capi()
    from sbo_b200 import workloads
    ds, lo, hi, pts, beta = workloads.small(d=d, pts_per_dim=ppd, n=n, seed=20 + d, G=G)
    engine.set_model(ds)
    engine.set_grid(lo, hi, pts)
    return beta, capi.UNSAFE_ANY if rule == "any" else capi.UNSAFE_ALL


def _fp64(engine, beta, rule):
    capi = _capi()
    engine.posterior(keep_v=capi.PRECISIONS["fp64"][1], fetch=False)
    engine.sets(beta, rule)
    return engine.expander(beta, None, capi.MODE_FANTASY, capi.PREC_FP64, want_counts=True)


@pytest.mark.parametrize("precision", ["tf32", "tf32x3"])
def test_cells_give_the_one_cell_counts(engine, precision):
    capi = _capi()
    prec, keep_v = capi.PRECISIONS[precision]
    cut_cases = 0
    for case in SMALL:
        beta, rule = _small(engine, *case)
        exact = _fp64(engine, beta, rule)
        engine.posterior(keep_v=keep_v, fetch=False)
        engine.sets(beta, rule)

        def run():
            return engine.expander(beta, None, capi.MODE_FANTASY, prec, want_counts=True)
        one = run()
        st1 = engine.refine_stats()
        if one["n_ambiguous"] == 0:                             # nothing inside the error bound: nothing refined
            assert st1 == {"cells": 0, "fp64_rows": 0}
            assert np.abs(one["counts"].astype(np.int64) - exact["counts"]).sum() <= 2
            continue
        assert st1["cells"] == 1 and st1["fp64_rows"] > 0, st1
        # aim at 3 x 3 cells; the 1 MB unit of the option and the 128-point floor of the posterior scratch bound how finely a
        # pass of a few hundred rows can be cut (7 to 16 cells measured on these cases; 179 rows fit 1 MB in one cell)
        mb, cut, st = _forced(engine, run, one, st1, min_cells=9)
        print(f"cells {precision} d={case[0]}: {one['n_ambiguous']} ambiguous pairs, one cell {st1['fp64_rows']} rows; "
              f"{mb} MB: {st['cells']} cells, {st['fp64_rows']} rows")
        if st["cells"] > 1:
            assert st["cells"] >= 4 and st["fp64_rows"] >= st1["fp64_rows"], (mb, st)
            cut_cases += 1
        assert np.array_equal(cut["counts"], one["counts"])
        for k in ("n_ambiguous", "n_refined_safe", "best_idx", "n_hit"):
            assert cut[k] == one[k], k
        assert np.abs(cut["counts"].astype(np.int64) - exact["counts"]).sum() <= 2
        st_auto = (run(), engine.refine_stats())[1]             # the option is back at 0: one cell again
        assert st_auto == st1
    assert cut_cases >= 1


def test_cells_after_a_list_overflow(engine):
    """fantasy_refine_cap = 16: the list overflows and the GEMM runs again with an exact list; that list is then refined
    cell by cell.  The counts must still be the one-cell (and FP64) ones."""
    capi = _capi()
    beta, rule = _small(engine, *SMALL[0])
    exact = _fp64(engine, beta, rule)
    prec, keep_v = capi.PRECISIONS["tf32"]
    engine.posterior(keep_v=keep_v, fetch=False)
    engine.sets(beta, rule)

    def run():
        return engine.expander(beta, None, capi.MODE_FANTASY, prec, want_counts=True)
    one = run()
    st1 = engine.refine_stats()
    try:
        engine.set_option("fantasy_refine_cap", 16)
        mb, cut, st = _forced(engine, run, one, st1, min_cells=4)
    finally:
        engine.set_option("fantasy_refine_cap", 0)
    assert cut["n_ambiguous"] > 16 and st["cells"] >= 4, st
    assert np.array_equal(cut["counts"], one["counts"])
    assert np.abs(cut["counts"].astype(np.int64) - exact["counts"]).sum() <= 2
    assert cut["best_idx"] == exact["best_idx"]


def test_a_budget_below_one_row_per_side_is_a_nomem_error(engine):
    """1 MB cannot hold the posterior scratch of even one point at n = 200, G = 4 (one 128-point chunk of 4 x 256 doubles):
    the library's NOMEM error names the option, and the context runs the next call normally."""
    capi = _capi()
    from sbo_b200.engine import SboError
    beta, rule = _small(engine, *SMALL[0])
    prec, keep_v = capi.PRECISIONS["tf32"]
    engine.posterior(keep_v=keep_v, fetch=False)
    engine.sets(beta, rule)
    before = engine.expander(beta, None, capi.MODE_FANTASY, prec, want_counts=True)
    try:
        engine.set_option("fantasy_refine_mb", 1)
        with pytest.raises(SboError, match="fantasy_refine_mb") as e:
            engine.expander(beta, None, capi.MODE_FANTASY, prec, want_counts=True)
        assert "error -4" in str(e.value)
    finally:
        engine.set_option("fantasy_refine_mb", 0)
    after = engine.expander(beta, None, capi.MODE_FANTASY, prec, want_counts=True)
    assert np.array_equal(after["counts"], before["counts"]) and after["best_idx"] == before["best_idx"]
    assert engine.refine_stats()["cells"] == 1
    with pytest.raises(ValueError):
        engine.set_option("fantasy_refine_mb", -1)


def test_c4_cells_give_the_default_counts(engine):
    capi = _capi()
    from sbo_b200 import workloads
    f = np.load(os.path.join(GOLD, "c4_full_sampled.npz"))
    ds, lo, hi, pts, beta = workloads.c4()
    engine.set_model(ds)
    engine.set_grid(lo, hi, pts)
    prec, keep_v = capi.PRECISIONS["tf32"]
    engine.posterior(keep_v=keep_v, fetch=False)
    engine.sets(beta, capi.UNSAFE_ALL)

    def run():
        return engine.expander(beta, None, capi.MODE_FANTASY, prec, want_counts=True)
    try:
        one = run()
        st1 = engine.refine_stats()
        mb, cut, st = _forced(engine, run, one, st1, min_cells=4, frac=1 / 8)
        print(f"C4 cells: {one['n_ambiguous']} ambiguous pairs, one cell {st1['fp64_rows']} rows; {mb} MB: {st['cells']} cells, "
              f"{st['fp64_rows']} rows; mem peak {engine.mem_peak() / 2 ** 30:.2f} GB")
    finally:
        engine.release(3)
    assert st1["cells"] == 1 and st["cells"] >= 4
    assert np.array_equal(cut["counts"], one["counts"])
    assert cut["n_hit"] == one["n_hit"] and cut["best_idx"] == one["best_idx"]
    assert np.array_equal(cut["counts"][f["x_idx"]].astype(np.int64), f["counts"])


def test_c5_model_cells_give_the_oracle_counts(engine):
    capi = _capi()
    spec = importlib.util.spec_from_file_location("make_fullsize_vectors", os.path.join(GOLD, "make_fullsize_vectors.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    f = np.load(os.path.join(GOLD, "c5_points_sampled.npz"))
    ds, beta, idx, P = mod.c5_sample_points()
    engine.set_model(ds)
    engine.set_points(P)
    prec, keep_v = capi.PRECISIONS["tf32"]
    engine.posterior(keep_v=keep_v, fetch=False)
    engine.sets(beta, capi.UNSAFE_ALL)

    def run():
        return engine.expander(beta, None, capi.MODE_FANTASY, prec, want_counts=True)
    try:
        one = run()
        st1 = engine.refine_stats()
        mb, cut, st = _forced(engine, run, one, st1, min_cells=4, frac=1 / 8)
        print(f"C5 model cells: {one['n_ambiguous']} ambiguous pairs, one cell {st1['fp64_rows']} rows; {mb} MB: {st['cells']} cells")
    finally:
        engine.release(3)
    assert st["cells"] >= 4
    xl = f["x_local"]
    assert np.array_equal(cut["counts"], one["counts"])
    assert np.array_equal(cut["counts"][xl].astype(np.int64), f["counts"])


def _bench(cmd, env=None):
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=900, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


@pytest.mark.parametrize("orchestrator", ["library", "torch"])
def test_two_gpus_with_cells_agree_with_one(engine, orchestrator):
    """The sharded step with the refinement cut into cells on every rank (SBO_FANTASY_REFINE_MB, read by GridEngine) against
    the single-GPU step with the automatic budget: same sets, expander size and x_new."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    capi = _capi()
    from sbo_b200 import workloads
    ds, lo, hi, pts, beta = workloads.c4(pts_per_dim=16, n=128)      # bench.py's c4s
    engine.set_model(ds)
    engine.set_grid(lo, hi, pts)
    prec, keep_v = capi.PRECISIONS["tf32"]
    engine.posterior(keep_v=keep_v, fetch=False)
    engine.sets(beta, capi.UNSAFE_ALL)

    def run():
        return engine.expander(beta, None, capi.MODE_FANTASY, prec, want_counts=True)
    one = run()
    mb, _, st = _forced(engine, run, one, engine.refine_stats(), min_cells=4)
    assert st["cells"] >= 4
    common = ["--workload", "c4s", "--mode", "fantasy", "--precision", "tf32", "--steps", "1", "--warmup", "1",
              "--no-cpu-baseline", "--no-peaks", "--no-reference-configs", "--no-lipschitz-steps"]
    ref = _bench([sys.executable, "bench.py"] + common)["config"]
    env = dict(os.environ, SBO_FANTASY_REFINE_MB=str(mb))
    two = _bench([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                  "--master-port", "29535", "bench.py", "--gpus", "2", "--orchestrator", orchestrator] + common, env)["config"]
    for k in ("n_safe", "n_unsafe", "n_min", "pairs", "n_hit", "x_new_idx"):
        assert ref[k] == two[k], k
