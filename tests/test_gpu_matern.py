"""GPU: Matern 3/2 and 5/2 models (sbo_set_model_ex) through the whole grid pipeline -- factorisation, posterior, gradients and
Lipschitz constants, the batched NLL, both pair tests, every fantasy precision and refinement mode, the drop-in classes and the
sharded steps -- against the kernel-parametrised NumPy reference tests/matern_ref.py and against the library's own FP64 kernels."""
import os
import sys

import numpy as np
import pytest

from conftest import ROOT, golden_ds
import matern_ref as R

pytestmark = pytest.mark.gpu
MATERN = ["Matern32", "Matern52"]
SMALL = [(3, 14, 70, 3, "all"), (4, 9, 200, 4, "any"), (6, 5, 130, 3, "any")]    # (d, points per axis, n, G, unsafe rule)
GOLD_CASES = [("c1", 9, 3.0, [48, 40], "all"), ("c3", 20, 2.0, [45, 61], "any")]
TF32_TOL = 1e-3                 # tests/test_gpu_parity.py: single-pass TF32 decisions vs FP64, in sf2 * (1 + gain) units


def _capi():
    from sbo_b200 import _capi
    return _capi


def _cases(request):
    from sbo_b200 import workloads
    out = []
    for d, ppd, n, G, rule in SMALL:
        ds, lo, hi, pts, beta = workloads.small(d=d, pts_per_dim=ppd, n=n, seed=30 + d, G=G)
        out.append((f"small d={d}", ds, lo, hi, pts, beta, rule))
    oracle = request.getfixturevalue("oracle")
    for name, n, beta, grid, rule in GOLD_CASES:
        gold = request.getfixturevalue(name)
        out.append((name, golden_ds(oracle, gold, n), gold["lo"], gold["hi"], grid, beta, rule))
    return out


def _rule(rule):
    capi = _capi()
    return capi.UNSAFE_ANY if rule == "any" else capi.UNSAFE_ALL


def _setup(engine, ds, lo, hi, grid, beta, rule, kernel, keep_v=0, with_grad=False):
    engine.set_model(ds, kernel)
    engine.set_grid(lo, hi, grid)
    mean, var = engine.posterior(with_grad=with_grad, keep_v=keep_v)
    engine.sets(beta, _rule(rule))
    return mean, var


def _near_x(margin, scale, tol):
    """per candidate: some pair within tol * scale of the threshold"""
    return (np.abs(margin) <= tol * scale).any(axis=0)


def _near_z(margin, scale, tol):
    return (np.abs(margin) <= tol * scale).any(axis=1)


def _scale(ds, var, S, beta, oracle):
    """band scale of a pair: sf2 * (1 + gain(x)) (tests/test_gpu_parity.py)"""
    d, G = ds["X_norm"].shape[1], var.shape[1]
    gain, sf2max = np.zeros(S.sum()), 0.0
    for i in range(1, G):
        _, sf2, sn2 = oracle.unpack_hyper(ds["hypopt"][:, i], d)
        sf2max = max(sf2max, sf2)
        vn = var[S, i] / ds["Y_std"][i] ** 2
        gain = np.maximum(gain, beta * np.sqrt(vn) / (vn + sn2 + oracle.EPS_F32))
    return sf2max * (1.0 + gain)[None, :]


# ---------------------------------------------------------------------------------------------------- model and posterior
@pytest.mark.parametrize("kernel", MATERN)
def test_model_posterior_gradient_and_lipschitz(engine, oracle, request, kernel):
    capi = _capi()
    for name, ds, lo, hi, grid, beta, rule in _cases(request):
        P = oracle.make_grid(lo, hi, grid)
        mean, var = _setup(engine, ds, lo, hi, grid, beta, rule, kernel, with_grad=True)
        fac = R.chol_factors(ds, kernel)
        mr, vr = R.posterior_chol(P, ds, kernel, factors=fac)
        n = ds["X_norm"].shape[0]
        L, W, a = engine.get_model()
        for i in range(ds["Y_norm"].shape[1]):
            assert np.max(np.abs(L[i] - fac[i][0])) <= 1e-10 * np.max(np.abs(fac[i][0])), name
            assert np.max(np.abs(a[i] - fac[i][1])) <= 1e-8 * np.max(np.abs(fac[i][1])), name
        assert np.max(np.abs(mean - mr)) <= 1e-10 * np.max(np.abs(mr)), name
        assert np.max(np.abs(var - vr)) <= 1e-10 * np.max(ds["Y_std"] ** 2 * np.exp(2 * ds["hypopt"][-2])), name
        sel = np.linspace(0, P.shape[0] - 1, 37).astype(int)
        pm, pv = engine.point_posterior(P[sel])
        assert np.max(np.abs(pm - mr[sel])) <= 1e-10 * np.max(np.abs(mr)) and np.max(np.abs(pv - vr[sel])) <= 1e-10 * np.max(vr)
        Lg = engine.lipschitz()
        for i in range(ds["Y_norm"].shape[1]):
            g = R.mean_grad(P, ds, i, kernel, factors=fac)
            assert Lg[i] == pytest.approx(np.max(np.abs(g)), rel=1e-9), (name, i)
            gp = engine.point_mean_grad(P[sel], i)
            assert np.max(np.abs(gp - g[sel])) <= 1e-9 * np.max(np.abs(g)), (name, i)
        assert n == engine.n
    assert capi.KERNELS[kernel] in (1, 2)


@pytest.mark.parametrize("kernel", MATERN)
def test_nll_batch_append_and_separable_options(engine, oracle, c3, kernel):
    from sbo_b200 import workloads
    rng = np.random.default_rng(4)
    Xn = c3["X"][:30]
    Xn = (Xn - Xn.mean(0)) / Xn.std(0)
    y = rng.normal(size=30)
    d = Xn.shape[1]
    H = np.column_stack([rng.uniform(-1.5, 1.5, size=(40, d + 1)), rng.uniform(-5, -2, size=40)])
    got = engine.nll_batch(Xn, y, H, kernel)
    want = np.array([R.negative_loglikelihood(h, Xn, y[:, None], kernel) for h in H])
    assert np.all(np.abs(got - want) <= 1e-9 * np.maximum(1.0, np.abs(want))), np.max(np.abs(got - want))
    # rank-1 appends across the 128-row padding boundary match the factorisation from scratch
    ds, lo, hi, pts, beta = workloads.small(d=3, pts_per_dim=10, n=132, seed=3, G=3)
    base = dict(ds)
    base["X_norm"], base["Y_norm"] = ds["X_norm"][:126], ds["Y_norm"][:126]
    engine.set_grid(lo, hi, pts)
    engine.set_model(base, kernel)
    for j in range(126, 132):
        engine.append_sample(ds["X_norm"][j], ds["Y_norm"][j])
    La, Wa, aa = engine.get_model()
    ma, va = engine.posterior()
    engine.set_model(ds, kernel)
    Lb, Wb, ab = engine.get_model()
    mb, vb = engine.posterior()
    assert np.max(np.abs(La - Lb)) <= 1e-11 * np.max(np.abs(Lb))
    assert np.max(np.abs(aa - ab)) <= 1e-8 * np.max(np.abs(ab))
    assert np.max(np.abs(ma - mb)) <= 1e-9 * np.max(np.abs(mb)) and np.max(np.abs(va - vb)) <= 1e-9 * np.max(ds["Y_std"]) ** 2
    # the separable SE-only options are ignored for a Matern model: the identical default path runs
    for opt in ("posterior_fused", "posterior_tables"):
        engine.set_option(opt, 1)
        try:
            m1, v1 = engine.posterior(with_grad=True)
        finally:
            engine.set_option(opt, 0)
        assert np.array_equal(m1, mb) and np.array_equal(v1, vb), opt
    with pytest.raises(ValueError):
        engine.set_model(ds, "Matern")


# ---------------------------------------------------------------------------------------------------- pair tests
@pytest.mark.parametrize("kernel", MATERN)
def test_lipschitz_steps_match_the_reference(engine, oracle, request, kernel):
    for name, ds, lo, hi, grid, beta, rule in _cases(request):
        P = oracle.make_grid(lo, hi, grid)
        engine.set_grid(lo, hi, grid)
        st = engine.safeopt_step(ds, beta, unsafe_rule=_rule(rule), kernel=kernel)
        so = R.safeopt_step(P, ds, beta, kernel, unsafe_rule=rule)
        assert st["n_safe"] == so["S"].sum() and st["n_unsafe"] == so["Z"].sum(), name
        assert st["x_new_idx"] == so["x_new_idx"], name
        gt = engine.goose_step(ds, beta, _rule(rule), kernel=kernel)
        go = R.goose_step(P, ds, beta, kernel, unsafe_rule=rule)
        assert (gt["target_idx"], gt["x_new_idx"], gt["explore_idx"]) == (go["target_idx"], go["x_new_idx"], go["explore_idx"]), name


@pytest.mark.parametrize("kernel", MATERN)
def test_fantasy_fp64_kernels_match_the_reference(engine, oracle, request, kernel):
    capi = _capi()
    for name, ds, lo, hi, grid, beta, rule in _cases(request):
        P = oracle.make_grid(lo, hi, grid)
        _setup(engine, ds, lo, hi, grid, beta, rule, kernel, keep_v=1)
        S, Z = engine.mask(capi.MASK_SAFE), engine.mask(capi.MASK_UNSAFE)
        cref, Tref = R.fantasy_pairs(P, ds, beta, S, Z, kernel)
        margin = R.fantasy_margin(P, ds, beta, S, Z, kernel)
        nx, nz = _near_x(margin, 1.0, 1e-9), _near_z(margin, 1.0, 1e-9)
        got = {}
        for var_, prune in ((1, 1), (0, 1), (1, 0), (0, 0)):
            engine.set_option("fantasy_f64_variant", var_)
            engine.set_option("fantasy_prune", prune)
            try:
                ex = engine.expander(beta, None, capi.MODE_FANTASY, capi.PREC_FP64, want_counts=True)
                tg = engine.goose_target(beta, None, capi.MODE_FANTASY, capi.PREC_FP64)
                T = engine.mask(capi.MASK_TARGET, 0)
            finally:
                engine.set_option("fantasy_f64_variant", 1)
                engine.set_option("fantasy_prune", 1)
            c = ex["counts"][S]
            got[(var_, prune)] = (c, T)
            dc = c != cref[S]
            dt = T != Tref
            print(f"{kernel} {name} f64 v{var_} prune {prune}: {int((c > 0).sum())} expanders, |T| {T.sum()}, "
                  f"{dc.sum()} counts / {dt.sum()} z differ ({nx.sum()} / {nz.sum()} near)")
            assert not (dc & ~nx).any() and not (dt[Z] & ~nz).any() and not dt[~Z].any(), (name, var_, prune)
            assert tg["n_hit"] == T.sum()
        for k, (c, T) in got.items():             # pruning on and off, SIMT and DMMA: equal FP64 counts
            assert np.array_equal(c, got[(1, 1)][0]) and np.array_equal(T, got[(1, 1)][1]), k


@pytest.mark.parametrize("kernel", MATERN)
@pytest.mark.parametrize("precision", ["tf32", "tf32x3"])
def test_refined_tensor_cores_give_the_fp64_sets(engine, oracle, request, kernel, precision):
    capi = _capi()
    for name, ds, lo, hi, grid, beta, rule in _cases(request):
        P = oracle.make_grid(lo, hi, grid)
        _setup(engine, ds, lo, hi, grid, beta, rule, kernel, keep_v=1)
        f64 = engine.expander(beta, None, capi.MODE_FANTASY, capi.PREC_FP64, want_counts=True)["counts"]
        engine.goose_target(beta, None, capi.MODE_FANTASY, capi.PREC_FP64)
        T64 = engine.mask(capi.MASK_TARGET, 0)
        mean, var = _setup(engine, ds, lo, hi, grid, beta, rule, kernel, keep_v=capi.PRECISIONS[precision][1])
        S, Z = engine.mask(capi.MASK_SAFE), engine.mask(capi.MASK_UNSAFE)
        ex = engine.expander(beta, None, capi.MODE_FANTASY, capi.PRECISIONS[precision][0], want_counts=True)
        tg = engine.goose_target(beta, None, capi.MODE_FANTASY, capi.PRECISIONS[precision][0])
        T = engine.mask(capi.MASK_TARGET, 0)
        margin = R.fantasy_margin(P, ds, beta, S, Z, kernel)
        scale = _scale(ds, var, S, beta, oracle)
        nx, nz = _near_x(margin, scale, 1e-12), _near_z(margin, scale, 1e-12)
        dc, dt = ex["counts"][S] != f64[S], (T != T64)[Z]
        print(f"{kernel} {precision} {name}: {ex['n_ambiguous']} ambiguous pairs, {ex['n_refined_safe']} refined safe; "
              f"{dc.sum()} counts / {dt.sum()} z differ from FP64; target {tg['n_ambiguous']} ambiguous")
        assert not (dc & ~nx).any() and not (dt & ~nz).any(), name
        # non-refining epilogue: TF32 against the TF32-operand emulation, TF32X3 against FP64
        engine.set_option("fantasy_refine", 0)
        try:
            raw = engine.expander(beta, None, capi.MODE_FANTASY, capi.PRECISIONS[precision][0], want_counts=True)
        finally:
            engine.set_option("fantasy_refine", 2)
        if precision == "tf32":
            ref32, _ = R.fantasy_pairs(P, ds, beta, S, Z, kernel, dtype="tf32")
            d0 = (raw["counts"][S] != ref32[S]) & ~_near_x(margin, scale, TF32_TOL)
        else:
            d0 = (raw["counts"][S] != f64[S]) & ~_near_x(margin, scale, 2e-5)
        assert not d0.any(), (name, int(d0.sum()))
        assert raw["n_ambiguous"] == 0


@pytest.mark.parametrize("kernel", MATERN)
def test_bounds_mode_and_forced_cells(engine, oracle, request, kernel):
    capi = _capi()
    for name, ds, lo, hi, grid, beta, rule in _cases(request)[:3]:
        _setup(engine, ds, lo, hi, grid, beta, rule, kernel, keep_v=2)
        S = engine.mask(capi.MASK_SAFE)
        exact = engine.expander(beta, None, capi.MODE_FANTASY, capi.PREC_TF32, want_counts=True)
        st1 = engine.refine_stats()
        engine.set_option("fantasy_refine", 3)
        try:
            bd = engine.expander(beta, None, capi.MODE_FANTASY, capi.PREC_TF32, want_counts=True)
        finally:
            engine.set_option("fantasy_refine", 2)
        c, cb = exact["counts"][S], bd["counts"][S]
        settled = cb >= 0
        assert np.all(cb[settled] <= c[settled])
        assert (c > 0).sum() <= bd["n_hit"] + bd["n_undecided"] and bd["n_hit"] <= (c > 0).sum()
        # budgets that cut the FP64 pass into cells give identical counts (down to the smallest budget that holds a pass)
        from sbo_b200.engine import SboError
        cells = []
        try:
            for mb in (64, 32, 16, 8, 4, 2, 1):
                engine.set_option("fantasy_refine_mb", mb)
                try:
                    cut = engine.expander(beta, None, capi.MODE_FANTASY, capi.PREC_TF32, want_counts=True)
                except SboError:
                    break
                cells.append(engine.refine_stats()["cells"])
                assert np.array_equal(cut["counts"], exact["counts"]) and cut["best_idx"] == exact["best_idx"], (name, mb)
        finally:
            engine.set_option("fantasy_refine_mb", 0)
        print(f"{kernel} {name}: one pass {st1}; cells per budget {cells}")
        assert cells


# ---------------------------------------------------------------------------------------------------- full size
def test_c4_matern52_default_counts_are_the_fp64_counts(engine):
    capi = _capi()
    from sbo_b200.engine import SboError
    from sbo_b200 import workloads
    ds, lo, hi, pts, beta = workloads.c4()
    kernel = "Matern52"
    engine.set_grid(lo, hi, pts)
    try:
        st = engine.safeopt_step(ds, beta, unsafe_rule=capi.UNSAFE_ALL, mode="fantasy", precision="tf32", kernel=kernel)
        S = engine.mask(capi.MASK_SAFE)
        c32 = engine.expander(beta, None, capi.MODE_FANTASY, capi.PREC_TF32, want_counts=True)["counts"]
        st1 = engine.refine_stats()
        # a budget that cuts the FP64 pass into at least 9 cells gives identical counts
        npad = (engine.n + 127) // 128 * 128
        mb, cut = max(1, int(st1["fp64_rows"] * (2 * engine.G - 1) * npad * 8 / 6 / 2 ** 20)), None
        try:
            while mb >= 1:
                engine.set_option("fantasy_refine_mb", mb)
                try:
                    r = engine.expander(beta, None, capi.MODE_FANTASY, capi.PREC_TF32, want_counts=True)
                except SboError:
                    break
                cut = (mb, r["counts"], engine.refine_stats())
                if cut[2]["cells"] >= 9:
                    break
                mb = min(mb - 1, mb * 3 // 4)
        finally:
            engine.set_option("fantasy_refine_mb", 0)
        gt32 = engine.goose_step(ds, beta, capi.UNSAFE_ALL, mode="fantasy", precision="tf32", upload=False)
        T32 = engine.mask(capi.MASK_TARGET, 0)
        st64 = engine.safeopt_step(ds, beta, unsafe_rule=capi.UNSAFE_ALL, mode="fantasy", precision="fp64", upload=False)
        c64 = engine.expander(beta, None, capi.MODE_FANTASY, capi.PREC_FP64, want_counts=True)["counts"]
        gt64 = engine.goose_step(ds, beta, capi.UNSAFE_ALL, mode="fantasy", precision="fp64", upload=False)
        T64 = engine.mask(capi.MASK_TARGET, 0)
        Z = engine.mask(capi.MASK_UNSAFE)
    finally:
        engine.release(3)
    diff = np.flatnonzero(c32 != c64)
    print(f"C4 {kernel}: |S| {S.sum()}, |Z| {Z.sum()}, {st['expander']['n_ambiguous']} ambiguous pairs, "
          f"{st['expander']['n_refined_safe']} refined safe, {int((c64 > 0).sum())} expanders, {diff.size} counts differ; "
          f"|T| {T32.sum()} / {T64.sum()}")
    print(f"C4 {kernel}: one pass {st1}; forced {cut[0]} MB: {cut[2]}")
    assert cut[2]["cells"] >= 9 and np.array_equal(cut[1], c32)
    assert diff.size == 0 and st["x_new_idx"] == st64["x_new_idx"]
    assert np.array_equal(T32, T64) and gt32["x_new_idx"] == gt64["x_new_idx"] and T64.sum() > 0
    # the DMMA counts against the NumPy reference: 32 candidates (both ragged ends, smallest / largest variance, spread)
    from oracle import gp_oracle as O
    P = O.make_grid(lo, hi, pts)
    xs, zs = np.flatnonzero(S), np.flatnonzero(Z)
    mean, var = R.posterior_chol(P[xs], ds, kernel)
    pick = np.unique(np.concatenate([xs[:4], xs[-4:], xs[np.argsort(var[:, 0])[:4]], xs[np.argsort(var[:, 0])[-4:]],
                                     xs[np.linspace(0, xs.size - 1, 24).astype(int)]]))
    assert pick.size >= 32
    ref = R.fantasy_counts_at(P[pick], P[zs], ds, beta, kernel)
    print(f"C4 {kernel} sampled: {pick.size} candidates, counts {ref[:8].tolist()} ...")
    assert np.array_equal(c64[pick], ref)


# ---------------------------------------------------------------------------------------------------- drop-in and sharded
def test_dropin_classes_follow_the_reference_decisions(oracle, c1):
    pkg = os.path.join(ROOT, "safe-bayesian-optimization_b200")
    if pkg not in sys.path:
        sys.path.insert(0, pkg)
    from models import GoOSE, SafeOpt
    from problems import Benoit_Problem as B
    from sbo_b200 import drivers
    bound = np.array([[-.6, 1.5], [-1., 1.]])
    P = oracle.make_grid(bound[:, 0], bound[:, 1], [100, 100])
    for algo, mode in (("safeopt", "lipschitz"), ("safeopt", "fantasy"), ("goose", "lipschitz"), ("goose", "fantasy")):
        plant = [B.Benoit_System_1, B.con1_system_tight]
        cls = SafeOpt if algo == "safeopt" else GoOSE
        bo = cls.BO(plant, bound, 3., grid_points_per_dim=100, expander_mode=mode, precision="tf32" if mode == "fantasy" else "fp64")
        bo.GP_initialization(c1["X"][:9], c1["Y"][:9], 'Matern52', multi_hyper=5, var_out=True, hypopt=c1["hyp_9"])
        seen = []

        def check(i, GP_m, x_new, y, info):
            ds = GP_m.inference_datasets
            ref = (R.safeopt_step if algo == "safeopt" else R.goose_step)(P, ds, 3., "Matern52", mode=mode)
            idx = ref["x_new_idx"]
            if idx < 0:                           # drivers.safeopt_iteration: the other candidate when one set is empty
                idx = max(ref["minimizer_idx"], ref["expander_idx"])
            np.testing.assert_array_equal(x_new, P[idx], err_msg=f"{algo} {mode} iteration {i}")
            seen.append(i)

        run = drivers.run_safeopt if algo == "safeopt" else drivers.run_goose
        kw = {"stop_std": -1.0} if algo == "safeopt" else {"f_opt": None}
        run(bo, n_iteration=3, on_iteration=check, hypopt=c1["hyp_9"], **kw)
        print(f"drop-in {algo} {mode} Matern52: {len(seen)} iterations, n = {bo.n_point}")
        assert seen == [0, 1, 2] and bo.kernel == 'Matern52'


def test_fit_on_device_reaches_the_host_optimum(c1):
    from sbo_b200.models.GP_Safe import GP
    X, Y = c1["X"][:14], c1["Y"][:14]
    for kernel in MATERN:
        host = GP([None, None]); host.hyper_seed = 5
        host.GP_initialization(X, Y, kernel, multi_hyper=5)
        dev = GP([None, None]); dev.hyper_seed = 5; dev.fit_on_device = True
        dev.GP_initialization(X, Y, kernel, multi_hyper=5)
        for i in range(2):
            a = host.negative_loglikelihood(host.hypopt[:, i], host.X_norm, host.Y_norm[:, i:i + 1])
            b = host.negative_loglikelihood(dev.hypopt[:, i], host.X_norm, host.Y_norm[:, i:i + 1])
            assert b <= a + 1e-3 * max(1.0, abs(a)), (kernel, i, a, b)


def test_one_rank_sharded_steps_equal_the_single_gpu_step(engine):
    import torch      # before the library loads NCCL
    import torch.distributed as dist
    import sbo_b200
    from sbo_b200 import sharded, workloads
    capi = _capi()
    ds, lo, hi, pts, beta = workloads.small(d=4, pts_per_dim=9, n=200, seed=34, G=4)
    own_group = not dist.is_initialized()
    if own_group:                      # the torch orchestrator: a one-process NCCL group
        dist.init_process_group("nccl", store=dist.HashStore(), rank=0, world_size=1, device_id=torch.device("cuda", 0))
    eng = sbo_b200.GridEngine(0)
    try:
        eng.set_grid(lo, hi, pts)
        engine.set_grid(lo, hi, pts)
        for kernel in MATERN:
            for mode, prec in (("lipschitz", "fp64"), ("fantasy", "tf32"), ("fantasy", "fp64")):
                one = engine.safeopt_step(ds, beta, unsafe_rule=capi.UNSAFE_ALL, mode=mode, precision=prec, kernel=kernel)
                tor = sharded.safeopt_step(eng, ds, beta, mode=mode, precision=prec, kernel=kernel)
                for k in ("x_new_idx", "expander_idx", "minimizer_idx", "n_safe", "n_unsafe"):
                    assert tor[k] == one[k], (kernel, mode, prec, k)
                g1 = engine.goose_step(ds, beta, capi.UNSAFE_ALL, mode=mode, precision=prec, kernel=kernel)
                gt = sharded.goose_step(eng, ds, beta, mode=mode, precision=prec, kernel=kernel)
                for k in ("target_idx", "x_new_idx", "explore_idx"):
                    assert gt[k] == g1[k], (kernel, mode, prec, k)
        eng.comm_init(0, 1, eng.comm_unique_id())
        for kernel in MATERN:
            for mode, prec in (("lipschitz", "fp64"), ("fantasy", "tf32")):
                one = engine.safeopt_step(ds, beta, unsafe_rule=capi.UNSAFE_ALL, mode=mode, precision=prec, kernel=kernel)
                lib = sharded.safeopt_step(eng, ds, beta, mode=mode, precision=prec, kernel=kernel)
                assert (lib["x_new_idx"], lib["n_safe"]) == (one["x_new_idx"], one["n_safe"]), (kernel, mode)
                g1 = engine.goose_step(ds, beta, capi.UNSAFE_ALL, mode=mode, precision=prec, kernel=kernel)
                gl = sharded.goose_step(eng, ds, beta, mode=mode, precision=prec, kernel=kernel)
                assert (gl["target_idx"], gl["x_new_idx"]) == (g1["target_idx"], g1["x_new_idx"]), (kernel, mode)
    finally:
        eng.close()
        if own_group:
            dist.destroy_process_group()


def test_two_gpus_agree_with_one():
    import json
    import subprocess
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29543", os.path.join("scripts", "matern_c4.py"), "--sharded-check"]
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=1800)
    assert r.returncode == 0, r.stderr[-3000:]
    out = json.loads(r.stdout.strip().splitlines()[-1])
    assert out["agree"], out
