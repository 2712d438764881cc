"""GPU: the incremental grid posterior (sbo_posterior_update) after sbo_append_sample, against sbo_posterior on the same
appended model (mean and Lipschitz constants bitwise, variance and new V-row entries to rounding), against the FP64 oracle on
the grown data set, over 40 chained updates, through every decision that reads the posterior, on shards, under the call-order
rules of the header, through the drop-in classes and at C4 size.

The grown data set keeps the normalisation of the first n0 samples (what sbo_append_sample holds): workloads.small with
n0 + m samples, of which the first n0 are installed and the other m appended."""
import ctypes as C

import numpy as np
import pytest

import matern_ref as R
from oracle import gp_oracle as O
from test_gpu_parity import TOL_CHOL, post_err

pytestmark = pytest.mark.gpu

VAR_TOL = 1e-12          # |var_update - var_posterior| <= VAR_TOL * sf2 * Y_std^2
DRIFT_TOL = 1e-11        # the same after 40 chained append + update cycles
V_TOL = 1e-12            # FP64 V rows: |dV| <= V_TOL * sqrt(sf2)
KERNELS = ("RBF", "Matern52")


def _capi():
    from sbo_b200 import _capi
    return _capi


@pytest.fixture(scope="module")
def eng():
    import sbo_b200
    e = sbo_b200.GridEngine(0)
    yield e
    e.close()


def _case(d, n0, m, seed=None):
    """(ds0, ds1, lo, hi, pts, beta): n0 installed samples and the grown set with m more, same normalisation."""
    from sbo_b200 import workloads
    pts = {2: 40, 3: 12, 4: 8, 6: 5}[d]
    ds1, lo, hi, pts, beta = workloads.small(d=d, pts_per_dim=pts, n=n0 + m, seed=seed if seed is not None else 30 + d, G=3)
    ds0 = dict(ds1, X_norm=ds1["X_norm"][:n0], Y_norm=ds1["Y_norm"][:n0])
    return ds0, ds1, lo, hi, pts, beta


def _append(eng, ds1, n0, n1):
    for r in range(n0, n1):
        eng.append_sample(ds1["X_norm"][r], ds1["Y_norm"][r])


def _scale(ds, i):
    d = ds["X_norm"].shape[1]
    _, sf2, _ = O.unpack_hyper(ds["hypopt"][:, i], d)
    return sf2, sf2 * ds["Y_std"][i] ** 2


def _check_var(ds, vu, vf, tol):
    for i in range(vu.shape[1]):
        err = np.max(np.abs(vu[:, i] - vf[:, i]))
        assert err <= tol * _scale(ds, i)[1], (i, err)


def _export(eng, beta, precision):
    """Safe candidates' exported V rows: (global index -> row) as (idx, rows[nx, G-1, len]) of float64 or uint32 words."""
    import torch
    capi = _capi()
    prec, _ = capi.PRECISIONS[precision]
    eng.sets(beta, capi.UNSAFE_ANY)
    info = eng.pairs_prepare(capi.MODE_FANTASY, prec, beta)
    nx, rd, vb = info["n_x_local"], info["row_doubles"], info["vrow_bytes"]
    assert nx > 0, "no candidates: the case does not exercise the V rows"
    rows = torch.zeros((nx, rd), dtype=torch.float64, device="cuda")
    vrows = torch.zeros((nx, vb), dtype=torch.uint8, device="cuda")
    eng.pairs_export(rows, vrows)
    torch.cuda.synchronize()
    v = vrows.cpu().numpy().view(np.float64 if precision == "fp64" else np.uint32).reshape(nx, eng.G - 1, -1)
    return rows.cpu().numpy()[:, -1].astype(np.int64), v


def _tf32_close(a_bits, b_bits, floor):
    """|a - b| <= one TF32 ulp of the larger magnitude, or <= floor (entries that are the result of cancellation carry the
    FP64 error of the sum, which the rounding to TF32 can turn into several ulps of a tiny value)."""
    a, b = a_bits.view(np.float32).astype(np.float64), b_bits.view(np.float32).astype(np.float64)
    ulp = np.spacing(np.maximum(np.abs(a), np.abs(b)).astype(np.float32)).astype(np.float64) * 8192.0
    diff = np.abs(a - b)
    return int(np.count_nonzero(a_bits != b_bits)), int(np.count_nonzero(diff > ulp)), bool(np.all((diff <= ulp) | (diff <= floor)))


def _check_vrows(ds, precision, n0, n1, exp0, exp_u, exp_f):
    """Kept V rows after the update: entries < n0 bitwise those of the n0-sample posterior, new ones as the recompute's."""
    idx0, V0 = exp0
    idx_u, Vu = exp_u
    idx_f, Vf = exp_f
    npad = Vu.shape[2] // (2 if precision == "tf32x3" else 1)
    npad0 = V0.shape[2] // (2 if precision == "tf32x3" else 1)        # smaller when the appends grew the padding
    common0, a0, b0 = np.intersect1d(idx_u, idx0, return_indices=True)
    assert common0.size > 0
    if precision == "tf32x3":
        assert np.array_equal(Vu[a0][:, :, :n0], V0[b0][:, :, :n0]) and np.array_equal(Vu[a0][:, :, npad:npad + n0], V0[b0][:, :, npad0:npad0 + n0])
    else:
        assert np.array_equal(Vu[a0][:, :, :n0], V0[b0][:, :, :n0])
    common, a, b = np.intersect1d(idx_u, idx_f, return_indices=True)
    assert common.size > 0
    report = []
    for c in range(Vu.shape[1]):
        sf2 = _scale(ds, c + 1)[0]
        u, f = Vu[a, c, n0:n1], Vf[b, c, n0:n1]
        if precision == "fp64":
            assert np.max(np.abs(u - f)) <= V_TOL * np.sqrt(sf2), c
        else:
            nd, nulp, ok = _tf32_close(u, f, V_TOL * np.sqrt(sf2))
            report.append((c, nd, nulp, u.size))
            assert ok, (c, nd, nulp)
            if precision == "tf32x3":       # the pair hi + lo carries ~FP32 accuracy
                hu = u.view(np.float32).astype(np.float64) + Vu[a, c, npad + n0:npad + n1].view(np.float32)
                hf = f.view(np.float32).astype(np.float64) + Vf[b, c, npad + n0:npad + n1].view(np.float32)
                assert np.max(np.abs(hu - hf)) <= 2.0 ** -20 * np.sqrt(sf2), c
    if report:
        print(f"{precision}: new V entries (constraint, differing, beyond 1 TF32 ulp, total) {report}")


# ------------------------------------------------------------------------------------------------
# 1 + 2: against sbo_posterior on the same appended model, and against the oracle on the grown data set
# ------------------------------------------------------------------------------------------------
EXPORT_BETA = 0.5        # the V rows are read through the candidate export; at beta = 2 the d = 6 cases have no safe point
@pytest.mark.parametrize("kind", ["mesh", "points"])
@pytest.mark.parametrize("kernel", KERNELS)
@pytest.mark.parametrize("d,n0,m", [(3, 40, 1), (3, 40, 17), (4, 40, 3), (4, 126, 6), (6, 40, 3), (6, 40, 17)])
def test_update_equals_posterior_on_the_appended_model(eng, d, n0, m, kernel, kind):
    ds0, ds1, lo, hi, pts, beta = _case(d, n0, m)
    n1 = n0 + m
    P = O.make_grid(lo, hi, pts)
    if kind == "mesh":
        eng.set_grid(lo, hi, pts)
    else:
        P = P[np.random.default_rng(d + m).permutation(P.shape[0])[:1500]]
        eng.set_points(P)
    grew = (n0 + 127) // 128 != (n1 + 127) // 128
    for kv, prec in ((0, None), (1, "fp64"), (2, "tf32"), (3, "tf32x3")):
        eng.set_model(ds0, kernel)
        eng.posterior(with_grad=kv == 0, keep_v=kv, fetch=False)
        exp0 = _export(eng, EXPORT_BETA, prec) if kv else None
        _append(eng, ds1, n0, n1)
        (mu, vu), info = eng.posterior_update()
        assert info == {"rows": m, "recomputed": bool(kv and grew)}
        Lu = eng.lipschitz() if kv == 0 else None
        exp_u = _export(eng, EXPORT_BETA, prec) if kv else None
        mf, vf = eng.posterior(with_grad=kv == 0, keep_v=kv)
        assert np.array_equal(mu, mf), kv
        _check_var(ds1, vu, vf, VAR_TOL)
        if kv == 0:
            assert np.array_equal(Lu, eng.lipschitz())
            # against the FP64 oracle on the grown data set
            mo, vo = R.posterior_chol(P, ds1, kernel)
            em, ev = post_err(O, ds1, mu, vu, mo, vo)
            assert em <= TOL_CHOL and ev <= TOL_CHOL, (em, ev)
        else:
            _check_vrows(ds1, prec, n0, n1, exp0, exp_u, _export(eng, EXPORT_BETA, prec))


# ------------------------------------------------------------------------------------------------
# 3: drift over chained updates
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kernel", KERNELS)
def test_forty_chained_updates_stay_within_tolerance(eng, kernel):
    ds0, ds1, lo, hi, pts, beta = _case(3, 30, 40)
    eng.set_grid(lo, hi, pts)
    eng.set_model(ds0, kernel)
    eng.posterior(with_grad=True, keep_v=2, fetch=False)
    for r in range(30, 70):
        eng.append_sample(ds1["X_norm"][r], ds1["Y_norm"][r])
        (mu, vu), info = eng.posterior_update()
        assert info["rows"] == 1 and not info["recomputed"]
    Lu = eng.lipschitz()
    mf, vf = eng.posterior(with_grad=True, keep_v=2)
    assert np.array_equal(mu, mf) and np.array_equal(Lu, eng.lipschitz())
    _check_var(ds1, vu, vf, DRIFT_TOL)


# ------------------------------------------------------------------------------------------------
# 4: every decision that reads the posterior
# ------------------------------------------------------------------------------------------------
def _decisions(eng, beta, mode, prec):
    capi = _capi()
    out = {}
    s = eng.sets(beta, capi.UNSAFE_ANY)
    out["sets"] = s
    out["masks"] = [eng.mask(k).copy() for k in (capi.MASK_SAFE, capi.MASK_MIN, capi.MASK_UNSAFE)]
    if mode == "lipschitz":
        Lg = eng.lipschitz()
        L = np.full(eng.G, Lg[eng.G - 1])
        ex = eng.expander(beta, L, capi.MODE_LIPSCHITZ, capi.PREC_FP64)
        out["exp_masks"] = [eng.mask(capi.MASK_EXPANDER, c) for c in range(eng.G - 1)]
    else:
        ex = eng.expander(beta, None, capi.MODE_FANTASY, prec, want_counts=True)
        out["counts"] = ex.pop("counts")
        out["exp_masks"] = [eng.mask(capi.MASK_EXPANDER, 0)]
    out["expander"] = ex
    std_min = np.sqrt(s["minimizer_var"]) if s["minimizer_idx"] >= 0 else 0.0
    std_exp = np.sqrt(ex["best_value"]) if ex["best_idx"] >= 0 else 0.0
    out["x_new"] = s["minimizer_idx"] if std_min > std_exp else ex["best_idx"]
    out["safeopt_batch"] = [p["idx"] for p in eng.safeopt_batch(4)]
    if mode == "lipschitz":
        tg = eng.goose_target(beta, L)
        out["tgt_masks"] = [eng.mask(capi.MASK_TARGET, c) for c in range(eng.G - 1)]
    else:
        tg = eng.goose_target(beta, None, capi.MODE_FANTASY, prec)
        out["tgt_masks"] = [eng.mask(capi.MASK_TARGET, 0)]
    out["target"] = tg
    out["goose_batch"] = [p["idx"] for p in eng.goose_batch(4)]
    return out


def _margins(mean, var, beta, tol=1e-10):
    """Grid points whose lcb or ucb lies within tol of a set threshold (0 for the constraints)."""
    lcb, ucb = mean - beta * np.sqrt(var), mean + beta * np.sqrt(var)
    near = (np.abs(lcb[:, 1:]) <= tol).any(axis=1) | (np.abs(ucb[:, 1:]) <= tol).any(axis=1)
    return np.flatnonzero(near)


@pytest.mark.parametrize("kernel", KERNELS)
@pytest.mark.parametrize("mode,prec", [("lipschitz", None), ("fantasy", "tf32"), ("fantasy", "tf32x3"), ("fantasy", "fp64")])
def test_decisions_after_the_update_equal_those_after_the_posterior(eng, kernel, mode, prec):
    capi = _capi()
    ds0, ds1, lo, hi, pts, beta = _case(4, 60, 3, seed=11)
    eng.set_grid(lo, hi, pts)
    p = capi.PRECISIONS[prec][0] if prec else capi.PREC_FP64
    kv = capi.PRECISIONS[prec][1] if prec else 0
    eng.set_model(ds0, kernel)
    eng.posterior(with_grad=True, keep_v=kv, fetch=False)
    _append(eng, ds1, 60, 63)
    (mu, vu), _ = eng.posterior_update()
    du = _decisions(eng, beta, mode, p)
    mf, vf = eng.posterior(with_grad=True, keep_v=kv)
    df = _decisions(eng, beta, mode, p)
    near = _margins(mf, vf, beta)
    assert du["sets"]["n_safe"] > 0 and du["expander"]["n_hit"] > 0, "the case does not exercise the pair stage"
    for k in du:
        assert _same(du[k], df[k]), f"{k} differs; points within 1e-10 of a threshold: {near.tolist()}"


# statistics of how the pair stage got to its result (tiles evaluated, pairs inside the TF32 error bound) may move with the
# last bits of the variance; the decisions may not
_WORK_KEYS = ("pairs_evaluated", "n_ambiguous", "n_refined_safe")


def _same(a, b):
    if isinstance(a, dict):
        return a.keys() == b.keys() and all(k in _WORK_KEYS or _same(a[k], b[k]) for k in a)
    if isinstance(a, (list, tuple)):
        return len(a) == len(b) and all(_same(x, y) for x, y in zip(a, b))
    if isinstance(a, np.ndarray):
        return np.array_equal(a, b)
    if isinstance(a, float):                  # values at a chosen point: var-derived, equal to rounding
        return a == b or abs(a - b) <= 1e-9 * max(abs(a), abs(b))
    return a == b


# ------------------------------------------------------------------------------------------------
# 5: shards, no collective
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shard", ["cyclic", "contiguous"])
def test_update_on_a_shard_equals_the_recompute_there(eng, shard):
    ds0, ds1, lo, hi, pts, beta = _case(3, 50, 5, seed=21)
    for kv in (0, 2):
        eng.set_grid(lo, hi, pts)
        if shard == "cyclic":
            eng.set_shard_cyclic(1, 3, 64)
        else:
            eng.set_shard(501, 603)
        eng.set_model(ds0, "RBF")
        eng.posterior(with_grad=kv == 0, keep_v=kv, fetch=False)
        _append(eng, ds1, 50, 55)
        (mu, vu), info = eng.posterior_update()
        assert info["rows"] == 5 and mu.shape[0] == eng.count
        Lu = eng.lipschitz() if kv == 0 else None
        mf, vf = eng.posterior(with_grad=kv == 0, keep_v=kv)
        assert np.array_equal(mu, mf)
        _check_var(ds1, vu, vf, VAR_TOL)
        if kv == 0:
            assert np.array_equal(Lu, eng.lipschitz())


# ------------------------------------------------------------------------------------------------
# 6: call order
# ------------------------------------------------------------------------------------------------
def _raw_update(eng):
    """sbo_posterior_update with NaN-filled host outputs: (rc, mean untouched, var untouched, launches during the call)."""
    capi = _capi()
    mean = np.full(eng.G * eng.count, np.nan)
    var = np.full(eng.G * eng.count, np.nan)
    info = capi.UpdateInfo()
    l0 = eng.kernel_launches()
    rc = eng._lib.sbo_posterior_update(eng._h, capi.dptr(mean), capi.dptr(var), C.byref(info))
    return rc, bool(np.isnan(mean).all()), bool(np.isnan(var).all()), eng.kernel_launches() - l0


def test_call_order_rules():
    import sbo_b200
    capi = _capi()
    ds0, ds1, lo, hi, pts, beta = _case(3, 40, 4, seed=3)
    e = sbo_b200.GridEngine(0)
    try:
        e.set_grid(lo, hi, pts)
        e.set_model(ds0)
        assert _raw_update(e) == (-1, True, True, 0)                              # no posterior at all
        invalidate = {
            "set_model": lambda: e.set_model(ds1),
            "set_model_ex": lambda: e.set_model(ds1, "Matern52"),
            "set_grid": lambda: e.set_grid(lo, hi, pts),
            "set_points": lambda: e.set_points(O.make_grid(lo, hi, pts)[:500]),
            "set_shard": lambda: e.set_shard(0, e.N),
            "set_shard_cyclic": lambda: e.set_shard_cyclic(0, 1, 64),
            "release_v": lambda: e.release(1),
        }
        for name, act in invalidate.items():
            e.set_grid(lo, hi, pts)
            e.set_model(ds0)
            e.posterior(keep_v=2 if name == "release_v" else 0, fetch=False)
            _append(e, ds1, 40, 42)
            act()
            assert _raw_update(e) == (-1, True, True, 0), name
            assert "sbo_posterior_update" in e._lib.sbo_last_error(e._h).decode()
        # releasing V rows that were never kept does not matter; m = 0 is a no-op that hands back the posterior
        e.set_grid(lo, hi, pts)
        e.set_model(ds0)
        m0, v0 = e.posterior(with_grad=True)
        e.release(1)
        l0 = e.kernel_launches()
        (m1, v1), info = e.posterior_update()
        assert info == {"rows": 0, "recomputed": False} and e.kernel_launches() == l0
        assert np.array_equal(m0, m1) and np.array_equal(v0, v1)
        _append(e, ds1, 40, 41)
        (_, _), info = e.posterior_update()
        assert info == {"rows": 1, "recomputed": False}
        # padding growth with V rows: the full posterior with the same flags, exactly
        dsg0, dsg1, lo2, hi2, pts2, beta2 = _case(3, 127, 3, seed=9)
        for kv in (0, 2):
            e.set_grid(lo2, hi2, pts2)
            e.set_model(dsg0)
            e.posterior(keep_v=kv, fetch=False)
            _append(e, dsg1, 127, 130)
            (mu, vu), info = e.posterior_update()
            assert info == {"rows": 3, "recomputed": kv != 0}
            mf, vf = e.posterior(keep_v=kv)
            assert np.array_equal(mu, mf)
            if kv:
                assert np.array_equal(vu, vf)
            else:
                _check_var(dsg1, vu, vf, VAR_TOL)
        ph = e.phase_ms()
        assert "posterior_update" in ph
    finally:
        e.close()


# ------------------------------------------------------------------------------------------------
# 7: the drop-in classes: step + add_sample_fixed
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("algo", ["safeopt", "goose"])
@pytest.mark.parametrize("mode", ["lipschitz", "fantasy"])
def test_dropin_fixed_model_loop_matches_full_steps(c3, algo, mode):
    import sbo_b200
    from sbo_b200 import drivers
    from sbo_b200.models import GoOSE, SafeOpt
    from sbo_b200.problems import WilliamOttoReactor_Problem
    wo = WilliamOttoReactor_Problem.WilliamOttoReactor()
    plant = [wo.get_objective, wo.get_constraint1, wo.get_constraint2]
    bound = np.array([[4., 7.], [70., 100.]])
    cls = SafeOpt.BO if algo == "safeopt" else GoOSE.BO
    bo = cls(plant, bound, 2., grid_points_per_dim=[60, 50], expander_mode=mode, precision="tf32")
    bo.GP_initialization(c3["X"][:20], c3["Y"][:20], 'RBF', multi_hyper=5, var_out=True, hypopt=c3["hyp_20"])
    ref = sbo_b200.GridEngine(0)
    launches = []
    upd = bo.engine.posterior_update

    def counted(*a, **k):
        l0 = bo.engine.kernel_launches()
        r = upd(*a, **k)
        launches.append((bo.engine.kernel_launches() - l0, r[1]["recomputed"]))
        return r

    bo.engine.posterior_update = counted
    try:
        ref.set_grid(bound[:, 0], bound[:, 1], [60, 50])
        for it in range(5):
            ds = dict(bo.inference_datasets)
            if algo == "safeopt":
                x_new, _ = drivers.safeopt_iteration(bo)
                r = ref.safeopt_step(ds, 2., mode=mode, precision="tf32")
            else:
                x_new, _ = drivers.goose_iteration(bo)
                r = ref.goose_step(ds, 2., mode=mode, precision="tf32")
            np.testing.assert_array_equal(x_new, ref.point_coords(r["x_new_idx"]), err_msg=f"iteration {it}")
            bo.add_sample_fixed(x_new, bo.calculate_plant_outputs(x_new, 0.))
    finally:
        ref.close()
    assert len(launches) == 4 and all(n <= 3 and not rec for n, rec in launches), launches


# ------------------------------------------------------------------------------------------------
# 8: C4 at full size
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("m", [1, 16])
def test_c4_full_size(eng, m):
    """The C4 recipe (32^4 grid, G = 4) with 513 installed samples: C4's own n = 512 fills its padded factor, so that any
    append would grow the padding and make the update recompute (kept V rows); from 513 up to 640 samples it does not."""
    from sbo_b200 import workloads
    capi = _capi()
    ds1, lo, hi, pts, beta = workloads.c4(n=513 + 16)
    ds = dict(ds1, X_norm=ds1["X_norm"][:513], Y_norm=ds1["Y_norm"][:513])
    prec, kv = capi.PRECISIONS["tf32"]
    eng.set_grid(lo, hi, pts)
    res = []
    for full in (False, True):
        eng.set_model(ds)
        eng.posterior(keep_v=kv, fetch=False)
        _append(eng, ds1, 513, 513 + m)
        if full:
            mv = eng.posterior(keep_v=kv)
        else:
            mv, info = eng.posterior_update()
            assert info == {"rows": m, "recomputed": False}
        s = eng.sets(beta)
        ex = eng.expander(beta, None, capi.MODE_FANTASY, prec)
        std_min = np.sqrt(s["minimizer_var"]) if s["minimizer_idx"] >= 0 else 0.0
        x_new = s["minimizer_idx"] if std_min > (np.sqrt(ex["best_value"]) if ex["best_idx"] >= 0 else 0.0) else ex["best_idx"]
        res.append((mv, eng.mask(capi.MASK_EXPANDER, 0), x_new, ex["n_hit"]))
    (mu, vu), Eu, xu, hu = res[0]
    (mf, vf), Ef, xf, hf = res[1]
    assert np.array_equal(mu, mf)
    _check_var(ds1, vu, vf, VAR_TOL)
    assert hu > 0 and np.array_equal(Eu, Ef) and xu == xf
