"""GPU: the fantasy-mode GoOSE target (column OR of the fantasy pair decisions, csrc/pairs.cu and csrc/fantasy_tc.cu) against
the NumPy reference (tests/goose_fantasy_ref.py) and against its own FP64 kernels, on one GPU and sharded."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch      # before the library loads NCCL (comm_init below): torch links its own NCCL build

from conftest import ROOT, golden_ds
from goose_fantasy_ref import goose_step_fantasy, goose_target_fantasy

pytestmark = pytest.mark.gpu
SMALL = [(4, 9, 200, 4, "any"), (3, 14, 70, 3, "all"), (6, 5, 130, 3, "any")]    # (d, points per axis, n, G, unsafe rule)
GOLD_CASES = [("c1", 9, 3.0, [48, 40], "all"), ("c3", 20, 2.0, [45, 61], "any")]
TF32_TOL = 1e-3                 # tests/test_gpu_parity.py: single-pass TF32 decisions vs FP64, in sf2 * (1 + gain) units


def _capi():
    from sbo_b200 import _capi
    return _capi


def _cases(request):
    """(ds, lo, hi, grid, beta, rule) of the small synthetic workloads and the C1 / C3 grids."""
    from sbo_b200 import workloads
    out = []
    for d, ppd, n, G, rule in SMALL:
        ds, lo, hi, pts, beta = workloads.small(d=d, pts_per_dim=ppd, n=n, seed=20 + d, G=G)
        out.append((f"small d={d}", ds, lo, hi, pts, beta, rule))
    oracle = request.getfixturevalue("oracle")
    for name, n, beta, grid, rule in GOLD_CASES:
        gold = request.getfixturevalue(name)
        out.append((name, golden_ds(oracle, gold, n), gold["lo"], gold["hi"], grid, beta, rule))
    return out


def _setup(engine, ds, lo, hi, grid, beta, rule, precision):
    capi = _capi()
    engine.set_model(ds)
    engine.set_grid(lo, hi, grid)
    mean, var = engine.posterior(keep_v=capi.PRECISIONS[precision][1])
    engine.sets(beta, capi.UNSAFE_ANY if rule == "any" else capi.UNSAFE_ALL)
    return mean, var


def _target(engine, beta, precision):
    capi = _capi()
    tg = engine.goose_target(beta, None, capi.MODE_FANTASY, capi.PRECISIONS[precision][0])
    return tg, engine.mask(capi.MASK_TARGET, 0)


def _reference(oracle, engine, ds, lo, hi, grid, beta, mean, var, dtype=np.float64):
    """Reference target on the engine's S and Z, the pair margins (|Z|,|S|) and the band scale sf2 * (1 + gain(x))."""
    capi = _capi()
    P = oracle.make_grid(lo, hi, grid)
    lcb, _ = oracle.bounds(mean, var, beta)
    S, Z = engine.mask(capi.MASK_SAFE), engine.mask(capi.MASK_UNSAFE)
    ref = goose_target_fantasy(P, ds, beta, S, Z, lcb, dtype=dtype)
    margin = np.abs(oracle.fantasy_margin(P, ds, beta, S, Z))
    d, G = P.shape[1], mean.shape[1]
    gain, sf2max = np.zeros(S.sum()), 0.0
    for i in range(1, G):
        _, sf2, sn2 = oracle.unpack_hyper(ds["hypopt"][:, i], d)
        sf2max = max(sf2max, sf2)
        vn = var[S, i] / ds["Y_std"][i] ** 2
        gain = np.maximum(gain, beta * np.sqrt(vn) / (vn + sn2 + oracle.EPS_F32))
    return ref, S, Z, margin, sf2max * (1.0 + gain)[None, :]


def _near(Z, margin, scale, tol):
    """z with at least one pair within tol * scale of the threshold (grid mask)."""
    out = np.zeros(Z.shape[0], dtype=bool)
    out[np.flatnonzero(Z)] = (margin <= tol * scale).any(axis=1)
    return out


@pytest.mark.parametrize("f64_variant", [1, 0])
def test_fp64_target_matches_the_reference(engine, oracle, request, f64_variant):
    capi = _capi()
    engine.set_option("fantasy_f64_variant", f64_variant)
    try:
        for name, ds, lo, hi, grid, beta, rule in _cases(request):
            mean, var = _setup(engine, ds, lo, hi, grid, beta, rule, "fp64")
            tg, T = _target(engine, beta, "fp64")
            ref, S, Z, margin, _ = _reference(oracle, engine, ds, lo, hi, grid, beta, mean, var)
            near = np.zeros(Z.shape[0], dtype=bool)
            near[np.flatnonzero(Z)] = (margin <= 1e-9).any(axis=1)
            diff = T != ref["mask"]
            print(f"fp64 v{f64_variant} {name}: |T| {T.sum()}, {near.sum()} z within 1e-9, {diff.sum()} differ")
            assert not (diff & ~near).any(), name
            assert tg["n_hit"] == T.sum() and tg["n_z"] == Z.sum() and tg["n_x"] == S.sum()
            assert tg["n_ambiguous"] == 0 and tg["n_refined_safe"] == 0
            if not diff.any():
                assert tg["best_idx"] == ref["best_idx"], name
                if tg["best_idx"] >= 0:
                    assert tg["best_value"] == pytest.approx(ref["best_lcb"], rel=1e-12, abs=1e-12)
                assert tg["per_idx"][0] == tg["best_idx"]
                st = engine.goose_step(ds, beta, capi.UNSAFE_ANY if rule == "any" else capi.UNSAFE_ALL, mode="fantasy",
                                       precision="fp64")
                so = goose_step_fantasy(oracle.make_grid(lo, hi, grid), ds, beta, rule)
                if np.array_equal(so["S"], S) and np.array_equal(so["Z"], Z):
                    assert (st["target_idx"], st["x_new_idx"], st["explore_idx"]) == \
                        (so["target_idx"], so["x_new_idx"], so["explore_idx"]), name
    finally:
        engine.set_option("fantasy_f64_variant", 1)


@pytest.mark.parametrize("precision", ["tf32", "tf32x3"])
def test_refined_tensor_cores_give_the_fp64_target(engine, oracle, request, precision):
    for name, ds, lo, hi, grid, beta, rule in _cases(request):
        mean, var = _setup(engine, ds, lo, hi, grid, beta, rule, precision)
        ref, S, Z, margin, scale = _reference(oracle, engine, ds, lo, hi, grid, beta, mean, var)
        for variant in (-1, 4, 6):             # auto; 2-CTA pairs with 4 / 8 epilogue warps (refinement forces 8)
            engine.set_option("fantasy_variant", variant)
            try:
                tg, T = _target(engine, beta, precision)
                engine.set_option("fantasy_refine", 0)
                raw, T0 = _target(engine, beta, precision)
            finally:
                engine.set_option("fantasy_refine", 2)
                engine.set_option("fantasy_variant", -1)
            near = _near(Z, margin, scale, 1e-12)
            diff = T != ref["mask"]
            print(f"{precision} v{variant} {name}: |T| {T.sum()} ({ref['mask'].sum()} fp64), {tg['n_ambiguous']} ambiguous pairs, "
                  f"{tg['n_refined_safe']} points added in FP64, {near.sum()} z within rounding, {diff.sum()} differ; "
                  f"refine 0: |T| {T0.sum()}")
            assert not (diff & ~near).any(), (name, variant)
            assert tg["n_hit"] == T.sum() and 0 <= tg["n_refined_safe"] <= tg["n_hit"]
            if not diff.any():
                assert tg["best_idx"] == ref["best_idx"], (name, variant)
            # the non-refining epilogue: the tensor-core decision stands (TF32: against the TF32-operand emulation)
            if precision == "tf32":
                ref32 = goose_target_fantasy(oracle.make_grid(lo, hi, grid), ds, beta, S, Z,
                                             oracle.bounds(mean, var, beta)[0], dtype="tf32")["mask"]
                d0 = (T0 != ref32) & ~_near(Z, margin, scale, TF32_TOL)
            else:
                d0 = (T0 != ref["mask"]) & ~_near(Z, margin, scale, 2e-5)
            assert not d0.any(), (name, variant, int(d0.sum()))
            assert raw["n_ambiguous"] == 0 and not T0[~Z].any()


def test_bounds_mode_brackets_the_fp64_target(engine, oracle, request):
    capi = _capi()
    for name, ds, lo, hi, grid, beta, rule in _cases(request):
        _setup(engine, ds, lo, hi, grid, beta, rule, "tf32")
        exact, Tx = _target(engine, beta, "tf32")
        engine.set_option("fantasy_refine", 3)
        try:
            bd, Tc = _target(engine, beta, "tf32")
        finally:
            engine.set_option("fantasy_refine", 2)
        print(f"bounds {name}: certified {bd['n_hit']}, undecided {bd['n_undecided']}, exact {exact['n_hit']}")
        assert not (Tc & ~Tx).any()                                   # certified subset of T
        assert Tx.sum() <= bd["n_hit"] + bd["n_undecided"]
        assert bd["n_hit"] == Tc.sum() and engine.refine_stats() == {"cells": 0, "fp64_rows": 0}
        if bd["n_undecided"] == 0:
            assert np.array_equal(Tc, Tx)
        else:
            assert bd["undecided_best_idx"] >= 0 and not Tc[bd["undecided_best_idx"]]
        if bd["undecided_best_value"] > bd["best_value"]:
            assert bd["best_idx"] == exact["best_idx"], name
        # the undecided z are exactly T's complement among them: T \ certified lies inside the undecided set
        added = Tx & ~Tc
        assert added.sum() <= bd["n_undecided"]
        assert capi.MASK_TARGET == 5


def test_list_overflow_and_the_filter(engine, oracle):
    """A list overflow gives the identical target; the filter (pairs whose z is already in T are dropped before the FP64 rows
    are planned) makes the target pass compute no more FP64 rows than the expander pass."""
    capi = _capi()
    from sbo_b200 import workloads
    d, ppd, n, G, rule = SMALL[0]
    ds, lo, hi, pts, beta = workloads.small(d=d, pts_per_dim=ppd, n=n, seed=20 + d, G=G)
    _setup(engine, ds, lo, hi, pts, beta, rule, "tf32")
    one, T1 = _target(engine, beta, "tf32")
    st1 = engine.refine_stats()
    engine.expander(beta, None, capi.MODE_FANTASY, capi.PREC_TF32)
    ste = engine.refine_stats()
    print(f"filter: target {one['n_ambiguous']} ambiguous pairs, {st1['fp64_rows']} FP64 rows; expander {ste['fp64_rows']} rows")
    assert st1["fp64_rows"] <= ste["fp64_rows"]
    try:
        engine.set_option("fantasy_refine_cap", 16)
        ov, Tov = _target(engine, beta, "tf32")
    finally:
        engine.set_option("fantasy_refine_cap", 0)
    assert ov["n_ambiguous"] > 16
    assert np.array_equal(Tov, T1) and ov["n_refined_safe"] == one["n_refined_safe"] and ov["best_idx"] == one["best_idx"]


def test_c4_default_target_is_the_fp64_dmma_target(engine):
    """C4 at full size: the default-mode target set is the FP64 (DMMA) one; a refinement budget that cuts the pass into at
    least 9 cells gives the identical set; the filtered target pass computes fewer FP64 rows than the expander's."""
    capi = _capi()
    from sbo_b200.engine import SboError
    from sbo_b200 import workloads
    ds, lo, hi, pts, beta = workloads.c4()
    engine.set_model(ds)
    engine.set_grid(lo, hi, pts)
    try:
        st32 = engine.goose_step(ds, beta, capi.UNSAFE_ALL, mode="fantasy", precision="tf32", upload=False)
        T32 = engine.mask(capi.MASK_TARGET, 0)
        st1 = engine.refine_stats()
        npad = (engine.n + 63) // 64 * 64
        mb, cut = max(1, int(st1["fp64_rows"] * (2 * engine.G - 1) * npad * 8 / 6 / 2 ** 20)), None
        try:
            while mb >= 1:
                engine.set_option("fantasy_refine_mb", mb)
                try:
                    r, T = _target(engine, beta, "tf32")
                except SboError:
                    break
                cut = (mb, r, T, engine.refine_stats())
                if cut[3]["cells"] >= 9:
                    break
                mb = min(mb - 1, mb * 3 // 4)
        finally:
            engine.set_option("fantasy_refine_mb", 0)
        engine.expander(beta, None, capi.MODE_FANTASY, capi.PREC_TF32)
        ste = engine.refine_stats()
        st64 = engine.goose_step(ds, beta, capi.UNSAFE_ALL, mode="fantasy", precision="fp64", upload=False)
        T64 = engine.mask(capi.MASK_TARGET, 0)
    finally:
        engine.release(3)
    print(f"C4 filter: target pass {st1}, expander pass {ste}; forced {cut[0]} MB: {cut[3]}")
    assert st1["fp64_rows"] <= ste["fp64_rows"]
    assert cut[3]["cells"] >= 9 and np.array_equal(cut[2], T32)
    assert cut[1]["best_idx"] == st32["target_idx"] and cut[1]["n_refined_safe"] == st32["target"]["n_refined_safe"]
    diff = np.flatnonzero(T32 != T64)
    print(f"C4 target: |T| tf32 {T32.sum()} fp64 {T64.sum()}, {st32['target']['n_ambiguous']} ambiguous pairs, "
          f"{st32['target']['n_refined_safe']} added in FP64, differing z {diff[:20].tolist()}")
    assert diff.size == 0
    for k in ("target_idx", "x_new_idx", "explore_idx", "n_safe", "n_unsafe"):
        assert st32[k] == st64[k], k
    assert st32["target"]["n_hit"] == T64.sum() > 0


def test_steps_sharded_and_dropin(engine, oracle, c1):
    capi = _capi()
    import sbo_b200
    from sbo_b200 import workloads
    d, ppd, n, G, rule = SMALL[1]
    ds, lo, hi, pts, beta = workloads.small(d=d, pts_per_dim=ppd, n=n, seed=20 + d, G=G)
    eng = sbo_b200.GridEngine(0)
    try:
        eng.set_grid(lo, hi, pts)
        eng.comm_init(0, 1, eng.comm_unique_id())
        engine.set_grid(lo, hi, pts)
        for prec in ("fp64", "tf32", "tf32x3"):
            one = engine.goose_step(ds, beta, capi.UNSAFE_ALL, mode="fantasy", precision=prec)
            sh = eng.goose_step_sharded(ds, beta, capi.UNSAFE_ALL, mode="fantasy", precision=prec)
            for k in ("target_idx", "target_lcb", "x_new_idx", "explore_idx", "n_safe", "n_unsafe", "min_lcb0_idx"):
                assert sh[k] == one[k], (prec, k)
            assert sh["target"]["n_hit"] == one["target"]["n_hit"]
        lip, lip1 = eng.goose_step_sharded(ds, beta, capi.UNSAFE_ALL), engine.goose_step(ds, beta, capi.UNSAFE_ALL)
        assert (lip["target_idx"], lip["x_new_idx"]) == (lip1["target_idx"], lip1["x_new_idx"])
    finally:
        eng.close()
    # the drop-in class on the Benoit problem (test/test_GoOSE.py setup): Target / explore_safeset agree with the engine's
    # fantasy step on the same model, and the reference driver completes 10 iterations
    pkg = os.path.join(ROOT, "safe-bayesian-optimization_b200")
    if pkg not in sys.path:
        sys.path.insert(0, pkg)
    from models import GoOSE
    from problems import Benoit_Problem as B
    from sbo_b200 import drivers
    plant = [B.Benoit_System_1, B.con1_system_tight]
    bound = np.array([[-.6, 1.5], [-1., 1.]])
    bo = GoOSE.BO(plant, bound, 3., grid_points_per_dim=100, expander_mode="fantasy", precision="tf32")
    bo.GP_initialization(c1["X"][:9], c1["Y"][:9], 'RBF', multi_hyper=5, var_out=True, hypopt=c1["hyp_9"])
    x_safe_min, min_safe_lcb = bo.minimize_obj_lcb()
    x_target, target_lcb = bo.Target()
    ref = sbo_b200.GridEngine(0)
    try:
        ref.set_grid(bound[:, 0], bound[:, 1], [100, 100])
        st = ref.goose_step(golden_ds(oracle, c1, 9), 3.0, capi.UNSAFE_ALL, mode="fantasy", precision="tf32")
        P = oracle.make_grid(bound[:, 0], bound[:, 1], [100, 100])
        assert st["target_idx"] >= 0
        np.testing.assert_array_equal(x_target, P[st["target_idx"]])
        assert target_lcb == st["target_lcb"]
        x_new = x_safe_min if min_safe_lcb <= target_lcb else bo.explore_safeset(x_target)
        np.testing.assert_array_equal(x_new, P[st["x_new_idx"]])
    finally:
        ref.close()
    data = drivers.run_goose(bo, n_iteration=10, f_opt=None, hypopt=c1["hyp_9"])
    print(f"drop-in fantasy GoOSE: last x {data['x_0'][-1]:.4f}, {data['x_1'][-1]:.4f}; objective {data['obj'][-1]:.4f}")
    assert len(data["i"]) == 10 and bo.n_point == 19


def _script(args, nproc=None):
    cmd = [sys.executable, os.path.join("scripts", "goose_fantasy.py")] + args
    if nproc:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(nproc), "--master-addr",
               "127.0.0.1", "--master-port", "29541", os.path.join("scripts", "goose_fantasy.py")] + args
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stderr[-3000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


@pytest.mark.parametrize("orchestrator", ["library", "torch"])
def test_two_gpus_agree_with_one(orchestrator):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    one = _script(["--workload", "c4s", "--sharded-reference"])
    two = _script(["--workload", "c4s", "--orchestrator", orchestrator, "--refine", "2"], nproc=2)
    for k in ("n_hit", "target_idx", "x_new_idx", "n_safe", "n_unsafe"):
        assert two[k] == one[k], k
    bd = _script(["--workload", "c4s", "--orchestrator", orchestrator, "--refine", "3"], nproc=2)
    assert bd["n_hit"] <= one["n_hit"] <= bd["n_hit"] + bd["n_undecided"]
