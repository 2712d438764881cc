"""GPU: the dimension and GP-count instantiations of the hot path that no other test runs (d = 1, 5, 7, 8 and G = 5 .. 8),
with a hyper-parameter table in which every entry differs, against the FP64 references.

The kernels are compiled once per input dimension and GP count the C ABI accepts (SBO_MAX_D = SBO_MAX_G = 8), and the
tensor-core fantasy records switch to 12 floats at d = 5.  workloads.synthetic sets ell = 1 in every dimension, sf2 = 1 and
one sn2 for every GP, so a kernel that reads the length-scale of the wrong dimension, or the sf2 / sn2 of the wrong GP,
computes the same numbers there.  Here every 1/2 log ell[k, g] is distinct, sf2 lies on both sides of 1 (log2 sf2 from -2
to 2, the terms of the tensor-core error bound) and sn2 differs per GP down to 4.5e-5 (large fantasy gains).  The grids
have a different point count per axis, so a mixed-up axis stride shows too.

The separable-table and fused posterior paths exist for the SE kernel only (a Matern model ignores those options), so they
run in the SE cases, d = 1, 4, 5, 7 and 8; at d = 3 and 6 they are not run here.

References: oracle/gp_oracle.py for the SE kernel, tests/matern_ref.py for Matern (its 'RBF' branch is the oracle's
arithmetic), tests/safeopt_batch_ref.py and tests/goose_batch_ref.py for the batch picks.  Tolerances and margin rules are
the ones of the tests named beside each stage.
"""
import functools
from types import SimpleNamespace

import numpy as np
import pytest

import matern_ref as R
import test_gpu_goose_batch as GBT
import test_gpu_safeopt_batch as SBT
from oracle import gp_oracle as O
from test_gpu_matern import _near_x, _near_z, _scale
from test_gpu_parity import TOL_CHOL, check_mask, post_err
from test_gpu_posterior_boundaries import LIP_REL, _check_lipschitz, _options, _reference

pytestmark = pytest.mark.gpu

# name -> (points per axis, n, G, kernel, unsafe rule, seed, r_train, constraint radii, half-width of the box around the
# training centre 0.3).  Together: every d in 1..8, every G in 2..8, n on both sides of the 128-row padding, both set paths
# (point count a multiple of 4 or not), SE and both Matern kernels.  Seeds, radii and boxes are chosen so that no stage is
# vacuous (asserted).
CASES = {
    "d1-G2-RBF": ([2001], 40, 2, "RBF", "all", 11, 0.9, (1.0,), 1.0),
    "d3-G4-Matern32": ([17, 16, 18], 129, 4, "Matern32", "any", 13, 0.9, (1.0, 1.1, 1.2), 1.0),
    "d4-G5-RBF": ([10, 9, 8, 9], 100, 5, "RBF", "any", 14, 0.9, (1.2, 1.3, 1.4, 1.5), 1.0),
    "d5-G6-RBF": ([7, 6, 6, 5, 6], 90, 6, "RBF", "any", 15, 1.4, (1.2, 1.3, 1.4, 1.5, 1.6), 0.7),
    "d6-G7-Matern52": ([4, 5, 4, 5, 4, 4], 70, 7, "Matern52", "any", 16, 1.4, (1.4, 1.5, 1.6, 1.7, 1.8, 1.9), 0.6),
    "d7-G8-RBF": ([4, 4, 3, 4, 4, 3, 4], 60, 8, "RBF", "any", 17, 1.8, (2.3, 2.4, 2.5, 2.6, 2.7, 2.8, 2.9), 0.4),
    "d8-G8-RBF": ([3] * 8, 60, 8, "RBF", "any", 18, 2.2, (2.6, 2.7, 2.8, 2.9, 3.0, 3.1, 3.2), 0.4),
}
LMULT = 1.25                     # pair-stage Lipschitz constants: 1.25 x each GP's own, so that not every safe point qualifies
Q = 4


def _capi():
    from sbo_b200 import _capi
    return _capi


def hyper_table(d, G, seed):
    """(d + 2, G) table with no two equal entries in a row block: 1/2 log ell over [-0.7, 0.7], 1/2 log sf2 over
    [-0.69, 0.69] (sf2 from 0.25 to 4), 1/2 log sn2 over [-5, -2] (the reference fit's bounds, GP_Safe.py:205-206)."""
    rng = np.random.default_rng(seed)
    hyp = np.empty((d + 2, G))
    hyp[:d] = rng.permutation(np.linspace(-0.7, 0.7, d * G)).reshape(d, G)
    hyp[d] = rng.permutation(np.linspace(-0.69, 0.69, G))
    hyp[d + 1] = rng.permutation(np.linspace(-5.0, -2.0, G))
    return hyp


@functools.lru_cache(maxsize=None)
def _case(name):
    """The case's data set, grid and FP64 reference factors / posterior on the grid (computed once per session)."""
    from sbo_b200 import workloads
    grid, n, G, kernel, rule, seed, r_train, radii, w = CASES[name]
    d = len(grid)
    ds, _, _, _, beta = workloads.synthetic(d, grid[0], n, seed, G, r_train=r_train, radii=radii)
    lo, hi = np.full(d, 0.3 - w), np.full(d, 0.3 + w)
    ds["hypopt"] = hyper_table(d, G, seed)
    P = O.make_grid(lo, hi, grid)
    fac, mean, var = _reference(O, P, ds, kernel)
    # a target with a different coordinate in every dimension (the distance and ball kernels take it as d scalars)
    target = lo + (hi - lo) * ((0.29 + 0.618034 * np.arange(d)) % 1.0)
    return SimpleNamespace(name=name, ds=ds, lo=lo, hi=hi, grid=grid, P=P, d=d, n=n, G=G, kernel=kernel, rule=rule,
                           beta=beta, seed=seed, fac=fac, mean=mean, var=var, target=target)


def _rule(c):
    capi = _capi()
    return capi.UNSAFE_ANY if c.rule == "any" else capi.UNSAFE_ALL


def _setup(engine, c, keep_v=0, with_grad=False):
    engine.set_model(c.ds, c.kernel)
    engine.set_grid(c.lo, c.hi, c.grid)
    m, v = engine.posterior(with_grad=with_grad, keep_v=keep_v)
    engine.sets(c.beta, _rule(c))
    return m, v


# ---------------------------------------------------------------------------------------------------- 1. model
@pytest.mark.parametrize("name", CASES)
def test_model_factors_and_appends(engine, name):
    """get_model against the reference Cholesky factors (test_gpu_parity.test_model_factorisation), and three rank-1
    appends against the factorisation of the grown set (test_gpu_matern.test_nll_batch_append_and_separable_options)."""
    c = _case(name)
    ds, n = c.ds, c.n
    engine.set_model(ds, c.kernel)
    L, W, alpha = engine.get_model()
    for i in range(c.G):
        Lo, ao = c.fac[i]
        K = R.build_K(ds["X_norm"], ds["hypopt"][:, i], c.kernel)
        assert np.max(np.abs(L[i] @ L[i].T - K)) <= 1e-12 * np.max(np.abs(K)), i
        assert np.max(np.abs(L[i] - Lo)) <= 1e-10 * np.max(np.abs(Lo)), i
        assert np.max(np.abs(W[i] @ Lo - np.eye(n))) <= 1e-9, i
        assert np.max(np.abs(alpha[i] - ao)) <= 1e-8 * max(1.0, np.max(np.abs(ao))), i
    base = dict(ds)
    base["X_norm"], base["Y_norm"] = ds["X_norm"][:n - 3], ds["Y_norm"][:n - 3]
    engine.set_grid(c.lo, c.hi, c.grid)
    engine.set_model(base, c.kernel)
    for j in range(n - 3, n):
        engine.append_sample(ds["X_norm"][j], ds["Y_norm"][j])
    La, _, aa = engine.get_model()
    ma, va = engine.posterior()
    engine.set_model(ds, c.kernel)
    Lb, _, ab = engine.get_model()
    mb, vb = engine.posterior()
    assert np.max(np.abs(La - Lb)) <= 1e-11 * np.max(np.abs(Lb))
    assert np.max(np.abs(aa - ab)) <= 1e-8 * np.max(np.abs(ab))
    assert np.max(np.abs(ma - mb)) <= 1e-9 * np.max(np.abs(mb)) and np.max(np.abs(va - vb)) <= 1e-9 * np.max(ds["Y_std"]) ** 2


# ---------------------------------------------------------------------------------------------------- 2. posterior
@pytest.mark.parametrize("name", CASES)
def test_grid_posterior_points_and_lipschitz(engine, name):
    """Grid mean / variance and every GP's Lipschitz constant on the default path and, for SE, on the separable factor
    tables and the fused table solve (test_gpu_posterior_boundaries); point_posterior and point_mean_grad off the grid."""
    c = _case(name)
    engine.set_model(c.ds, c.kernel)
    engine.set_grid(c.lo, c.hi, c.grid)
    paths = [{}] + ([{"posterior_tables": 1}, {"posterior_fused": 1}] if c.kernel == "RBF" else [])
    for opts in paths:
        with _options(engine, **opts):
            m, v = engine.posterior(with_grad=True)
            L = engine.lipschitz()
        em, ev = post_err(O, c.ds, m, v, c.mean, c.var)
        assert em <= TOL_CHOL and ev <= TOL_CHOL, (opts, em, ev)
        _check_lipschitz(L, c.P, c.ds, c.kernel, c.fac)
    X = np.random.default_rng(c.seed).uniform(c.lo, c.hi, size=(64, c.d))
    pm, pv = engine.point_posterior(X)
    _, mo, vo = _reference(O, X, c.ds, c.kernel)
    em, ev = post_err(O, c.ds, pm, pv, mo, vo)
    assert em <= TOL_CHOL and ev <= TOL_CHOL, (em, ev)
    for i in range(c.G):
        g = engine.point_mean_grad(X, i)
        go = R.mean_grad(X, c.ds, i, c.kernel, factors=c.fac)
        assert np.max(np.abs(g - go)) <= LIP_REL * np.max(np.abs(go)), i


# ---------------------------------------------------------------------------------------------------- 3. sets
@pytest.mark.parametrize("name", CASES)
def test_sets_argreduce_and_ball(engine, name):
    """Pass 1 and pass 2 (test_gpu_parity.test_sets_full_grid): S and Z against the reference posterior up to points within
    SET_TOL of a threshold, every result field and the S / Z / M masks exactly from the GPU's own posterior; then the
    nearest safe point to a d-dimensional target and the safe points in a ball around it."""
    capi = _capi()
    c = _case(name)
    engine.set_model(c.ds, c.kernel)
    engine.set_grid(c.lo, c.hi, c.grid)
    m, v = engine.posterior()
    s1 = engine.sets_pass1(c.beta, _rule(c))
    s2 = engine.sets_pass2(s1["min_ucb0"])
    S, Z, M = (engine.mask(k) for k in (capi.MASK_SAFE, capi.MASK_UNSAFE, capi.MASK_MIN))
    N = c.P.shape[0]
    assert 0 < s1["n_safe"] < N and s1["n_unsafe"] > 0, s1
    lcb, _ = O.bounds(c.mean, c.var, c.beta)
    cmargin = np.min(np.abs(lcb[:, 1:]), axis=1)
    scale = float(np.max(c.ds["Y_std"][1:]))
    check_mask(S, O.safe_mask(lcb), cmargin, scale, "S")
    check_mask(Z, O.unsafe_mask(lcb, c.rule), cmargin, scale, "Z")
    lg, ug = O.bounds(m, v, c.beta)
    assert np.array_equal(S, O.safe_mask(lg)) and np.array_equal(Z, O.unsafe_mask(lg, c.rule))
    i_u, v_u = O.minimize_obj_ucb(ug, S)
    i_l, v_l = O.minimize_obj_lcb(lg, S)
    mi, _, Mo, _ = O.minimizer(v, lg, ug, S)
    want1 = {"n_safe": S.sum(), "n_unsafe": Z.sum(), "min_ucb0": v_u, "min_ucb0_idx": i_u, "min_lcb0": v_l, "min_lcb0_idx": i_l,
             "n_min": 0, "minimizer_var": -np.inf, "minimizer_idx": -1}
    assert s1 == want1, (s1, want1)
    want2 = dict(want1, n_min=Mo.sum(), minimizer_var=v[mi, 0], minimizer_idx=mi)
    assert s2 == want2, (s2, want2)
    assert np.array_equal(M, Mo) and Mo.any()
    assert engine.sets(c.beta, _rule(c)) == want2
    # nearest safe point (test_gpu_parity.test_user_mask_argreductions) and the trust-region ball
    idx, dist = engine.argreduce(capi.ARGMIN_DIST, capi.MASK_SAFE, 0, c.target)
    io, do = O.explore_safeset(c.P, S, c.target)
    assert idx == io and dist == pytest.approx(do, rel=1e-14)
    dall = np.linalg.norm(c.P - c.target, axis=1)
    ds_ = np.unique(dall[S])
    r = 0.5 * (ds_[ds_.size // 2] + ds_[ds_.size // 2 + 1])         # halfway between two distances of safe points
    engine.user_mask_ball(c.target, r, capi.MASK_SAFE)
    U = engine.mask(capi.MASK_USER)
    want = S & (dall <= r)
    bad = U != want
    assert np.all(np.abs(dall[bad] - r) <= 1e-12 * r), int(bad.sum())
    assert 0 < U.sum() < S.sum()


# ---------------------------------------------------------------------------------------------------- 4. Lipschitz pairs
@pytest.mark.parametrize("name", CASES)
def test_lipschitz_pair_stage(engine, name):
    """Expander and GoOSE target with a different L per constraint against the all-pairs reference, culled and un-culled
    (test_gpu_parity.test_expander_and_target_lipschitz and test_tile_culling_is_exact)."""
    capi = _capi()
    c = _case(name)
    m, v = _setup(engine, c, with_grad=True)
    S, Z = engine.mask(capi.MASK_SAFE), engine.mask(capi.MASK_UNSAFE)
    lcb, ucb = O.bounds(m, v, c.beta)
    L = engine.lipschitz() * LMULT                 # one constant per GP: the GPs' hyper-parameters all differ
    assert np.unique(L[1:]).size == c.G - 1
    exo = O.expander_lipschitz(c.P, S, Z, ucb, v, L)
    tgo = O.goose_target(c.P, S, Z, ucb, lcb, L)
    assert exo["masks"].any() and tgo["masks"].any()
    res = {}
    try:
        for cull in (1, 0):
            engine.set_option("pair_cull", cull)
            ex = engine.expander(c.beta, L)
            em = [engine.mask(capi.MASK_EXPANDER, k) for k in range(c.G - 1)]
            tg = engine.goose_target(c.beta, L)
            tm = [engine.mask(capi.MASK_TARGET, k) for k in range(c.G - 1)]
            res[cull] = (ex, em, tg, tm)
    finally:
        engine.set_option("pair_cull", 1)
    ex, em, tg, tm = res[1]
    for k in range(c.G - 1):
        assert (em[k] != exo["masks"][k]).sum() <= 2, k            # only exact-threshold rounding may differ
        assert (tm[k] != tgo["masks"][k]).sum() <= 2, k
    assert ex["n_x"] == S.sum() and ex["n_z"] == Z.sum() and ex["pairs_algorithmic"] == S.sum() * Z.sum() * (c.G - 1)
    if all(np.array_equal(em[k], exo["masks"][k]) for k in range(c.G - 1)):
        assert ex["best_idx"] == exo["best_idx"] and ex["per_idx"] == [p for p, _ in exo["per_idx"]]
        assert np.sqrt(ex["best_value"]) == pytest.approx(exo["best_std"], rel=1e-12)
    if all(np.array_equal(tm[k], tgo["masks"][k]) for k in range(c.G - 1)):
        assert tg["best_idx"] == tgo["best_idx"] and tg["best_value"] == tgo["best_lcb"]
    ex0, em0, tg0, tm0 = res[0]
    for k in range(c.G - 1):
        assert np.array_equal(em0[k], em[k]) and np.array_equal(tm0[k], tm[k]), k
    for key in ("best_idx", "best_value", "per_idx", "per_value", "n_hit", "pairs_algorithmic"):
        assert ex0[key] == ex[key] and tg0[key] == tg[key], key


# ---------------------------------------------------------------------------------------------------- 5. fantasy pairs
def _fantasy(engine, c, precision, goose_too=True):
    capi = _capi()
    prec, keep_v = capi.PRECISIONS[precision]
    _setup(engine, c, keep_v=keep_v)
    ex = engine.expander(c.beta, None, capi.MODE_FANTASY, prec, want_counts=True)
    if not goose_too:
        return ex, None, None
    tg = engine.goose_target(c.beta, None, capi.MODE_FANTASY, prec)
    return ex, tg, engine.mask(capi.MASK_TARGET, 0)


@pytest.mark.parametrize("name", CASES)
def test_fantasy_pair_stage(engine, name):
    """FP64 counts and target (DMMA and SIMT) against the reference up to pairs within 1e-9 of the threshold
    (test_gpu_matern.test_fantasy_fp64_kernels_match_the_reference); refined TF32 / TF32X3 counts and target equal to the
    FP64 ones up to pairs within 1e-12 sf2 (1 + gain) (test_gpu_parity._fantasy_tc_case); bounds mode brackets the FP64
    expander set (test_gpu_prune.test_bounds_mode_brackets_the_fp64_expander_set)."""
    capi = _capi()
    c = _case(name)
    m, v = _setup(engine, c, keep_v=1)
    S, Z = engine.mask(capi.MASK_SAFE), engine.mask(capi.MASK_UNSAFE)
    cref, Tref = R.fantasy_pairs(c.P, c.ds, c.beta, S, Z, c.kernel)
    margin = R.fantasy_margin(c.P, c.ds, c.beta, S, Z, c.kernel)
    assert (cref[S] > 0).any() and Tref.any(), "no fantasy expander member or target"
    nx, nz = _near_x(margin, 1.0, 1e-9), _near_z(margin, 1.0, 1e-9)
    got = {}
    try:
        for variant in (1, 0):
            engine.set_option("fantasy_f64_variant", variant)
            ex, tg, T = _fantasy(engine, c, "fp64")
            dc, dt = ex["counts"][S] != cref[S], T != Tref
            assert not (dc & ~nx).any() and not (dt[Z] & ~nz).any() and not dt[~Z].any(), (variant, int(dc.sum()), int(dt.sum()))
            assert (ex["counts"][~S] == 0).all() and tg["n_hit"] == T.sum()
            assert ex["pairs_algorithmic"] == S.sum() * Z.sum() * (c.G - 1)
            got[variant] = (ex["counts"], T)
    finally:
        engine.set_option("fantasy_f64_variant", 1)
    assert np.array_equal(got[0][0], got[1][0]) and np.array_equal(got[0][1], got[1][1])
    c64, T64 = got[1]
    # refined tensor cores: the FP64 counts and target
    scale = _scale(c.ds, v, S, c.beta, O)
    exact = (np.abs(margin) <= 1e-12 * scale).sum(axis=0)
    near_z = _near_z(margin, scale, 1e-12)
    for precision in ("tf32", "tf32x3"):
        ex, tg, T = _fantasy(engine, c, precision)
        dr = np.abs(ex["counts"][S].astype(np.int64) - cref[S])
        assert np.all(dr <= exact), (precision, int(dr.max()), int((dr > exact).sum()))
        assert (ex["counts"][~S] == 0).all()
        dt = T != T64
        assert not (dt[Z] & ~near_z).any() and not dt[~Z].any(), (precision, int(dt.sum()))
        print(f"{name} {precision}: {ex['n_ambiguous']} ambiguous pairs, {ex['n_refined_safe']} refined safe, "
              f"{int((c64 > 0).sum())} expanders, |T| {T.sum()}")
    # bounds mode: certified <= FP64 <= certified + undecided
    try:
        engine.set_option("fantasy_refine", 3)
        bd, _, _ = _fantasy(engine, c, "tf32", goose_too=False)
    finally:
        engine.set_option("fantasy_refine", 2)
    cb, und = bd["counts"], bd["counts"] < 0
    assert (cb > 0).any(), "bounds mode certified no candidate: the bracket says nothing"
    assert np.all(cb[~und] <= c64[~und])
    assert np.all(c64[cb > 0] > 0) and np.all((cb > 0) | und | (c64 == 0))
    assert bd["n_hit"] == int((cb > 0).sum()) and bd["n_undecided"] == int(und.sum())


# ---------------------------------------------------------------------------------------------------- 6. batch picks
@pytest.mark.parametrize("name", CASES)
def test_batch_picks(engine, name):
    """q = 4 SafeOpt and GoOSE batch picks after a Lipschitz step against the NumPy references (test_gpu_safeopt_batch,
    test_gpu_goose_batch): the hallucinated downdates read the objective's length-scales, anisotropic here."""
    c = _case(name)
    engine.set_grid(c.lo, c.hi, c.grid)
    st = engine.safeopt_step(c.ds, c.beta, unsafe_rule=_rule(c), kernel=c.kernel)
    state = SBT._state(engine)
    picks = engine.safeopt_batch(Q)
    assert len(picks) == Q and picks[0]["idx"] == (st["x_new_idx"] if st["x_new_idx"] >= 0 else st["minimizer_idx"])
    SBT._compare(picks, SBT._reference(engine, c.ds, c.lo, c.hi, c.grid, c.kernel, state, Q, [p["idx"] for p in picks]), name)
    gs = engine.goose_step(c.ds, c.beta, _rule(c), kernel=c.kernel)
    gstate = GBT._state(engine)
    gpicks = engine.goose_batch(Q)
    assert len(gpicks) == Q
    GBT._check_pick_one(gpicks, gs)
    GBT._compare(gpicks, GBT._reference(c.ds, c.lo, c.hi, c.grid, c.beta, c.kernel, gstate, Q, GBT._forced(gpicks)), name)


# ---------------------------------------------------------------------------------------------------- 7. NLL
@pytest.mark.parametrize("kernel", R.KERNELS)
@pytest.mark.parametrize("name", [k for k in CASES if len(CASES[k][0]) in (1, 5, 7, 8)])
def test_nll_batch(engine, name, kernel):
    """sbo_nll_batch for 8 hyper-parameter vectors inside the fit's bounds (test_gpu_dropin.test_batched_nll_matches_oracle)."""
    c = _case(name)
    rng = np.random.default_rng(c.seed)
    Xn, y = c.ds["X_norm"], c.ds["Y_norm"][:, 1]
    H = np.column_stack([rng.uniform(-1.5, 1.5, size=(8, c.d + 1)), rng.uniform(-5.0, -2.0, size=8)])
    got = engine.nll_batch(Xn, y, H, kernel)
    want = np.array([O.negative_loglikelihood(h, Xn, y[:, None]) if kernel == "RBF" else
                     R.negative_loglikelihood(h, Xn, y[:, None], kernel) for h in H])
    assert np.all(np.abs(got - want) <= 1e-9 * np.maximum(1.0, np.abs(want))), np.max(np.abs(got - want))
