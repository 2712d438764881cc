"""GPU: the grid posterior where its loop and offset logic does something -- training sizes on both sides of the 128-row
blocks of the solve, several chunks with a ragged last one, contiguous shards with unaligned cut points, the V rows the
posterior keeps for the fantasy expander and the candidate rows it exports, and the solve paths the options select.

References: the FP64 oracle (oracle.chol_factors / posterior_chol, V = L^-1 k(X, x)) for the SE kernel and
tests/matern_ref.py for Matern 5/2.  Where the per-point arithmetic cannot depend on the layout (chunk size, shard cut,
keep_v, explicit points vs grid), the comparison is bitwise."""
import contextlib

import numpy as np
import pytest

import matern_ref as R
from conftest import load_golden
from oracle.gp_oracle import round_tf32
from test_gpu_parity import TOL_CHOL, post_err

pytestmark = pytest.mark.gpu

N_LIST = [2, 64, 65, 127, 128, 129, 255, 256, 257]    # n = 1 has no X_std: 2 is the smallest model the normalisation accepts
LIP_REL = 1e-9                                         # Lipschitz constants, as test_gpu_parity.test_mean_gradient_and_lipschitz
V_TOL = 1e-12                                          # FP64 V rows: |dV| <= V_TOL * sqrt(sf2)
AB_REL = 1e-12                                         # exported fantasy gains a, b
DEFAULTS = {"posterior_chunk_mb": 0, "posterior_variant": 1, "posterior_tables": 0, "posterior_fused": 0}
GRIDS = {"c3": [41, 37], "d3": [13, 13, 13], "d4": [7, 7, 7, 7]}                   # odd sizes: ragged last CTA
BIG = {"c3": [173, 181], "d3": [31, 31, 31], "d4": [13, 13, 13, 13]}               # 31313 / 29791 / 28561 points


def _capi():
    from sbo_b200 import _capi
    return _capi


@contextlib.contextmanager
def _options(engine, **kw):
    """Set posterior options on the shared engine; restore what it had before, whatever happens."""
    before = {k: engine.options.get(k, DEFAULTS[k]) for k in kw}
    try:
        for k, v in kw.items():
            engine.set_option(k, v)
        yield
    finally:
        for k, v in before.items():
            engine.set_option(k, v)


def _case(name, n):
    """(ds, lo, hi, beta): the golden C3 set (d = 2, G = 3; beyond its 35 points the recipe of test_model_factorisation)
    or workloads.small at d = 3, G = 2 and d = 4, G = 4."""
    from oracle import gp_oracle as O
    if name == "c3":
        c3 = load_golden("c3_wor")
        if n <= 35:
            X, Y, hyp = c3["X"][:n], c3["Y"][:n], c3[f"hyp_{5 if n <= 5 else (20 if n <= 20 else 35)}"]
        else:
            X = np.random.default_rng(n).uniform([4, 70], [7, 100], size=(n, 2))
            Y = np.column_stack([np.sin(X[:, 0]) * X[:, 1], 0.1 - 0.01 * X[:, 0], 0.05 + 0.001 * X[:, 1]])
            hyp = c3["hyp_35"]
        return O.make_inference_datasets(X, Y, hyp, with_inverse=False), c3["lo"], c3["hi"], 2.0
    from sbo_b200 import workloads
    d = int(name[1])
    ds, lo, hi, _, beta = workloads.small(d=d, n=n, seed=40 + d, G=2 if d == 3 else 4)
    return ds, lo, hi, beta


def _reference(oracle, P, ds, kernel, return_V=False):
    """(factors, mean, var[, V rows]) of the Cholesky-form reference for the covariance function `kernel`."""
    if kernel == "RBF":
        fac = oracle.chol_factors(ds)
        return (fac,) + tuple(oracle.posterior_chol(P, ds, return_V=return_V, factors=fac))
    fac = R.chol_factors(ds, kernel)
    return (fac,) + tuple(R.posterior_chol(P, ds, kernel, return_V=return_V, factors=fac))


def _check_lipschitz(L, P, ds, kernel, fac):
    for i in range(ds["Y_norm"].shape[1]):
        assert L[i] == pytest.approx(R.lipschitz_constant(P, ds, i, kernel, factors=fac), rel=LIP_REL), i


def _npad(n):
    return -(-n // 128) * 128


def _export(engine, beta, precision):
    """sets -> pairs_prepare(FANTASY, precision) -> pairs_export into torch CUDA tensors.  Returns the exported rows
    [n_x, row_doubles] and the V rows [n_x, G-1, row length] (float64 for fp64, float32 bit patterns for tf32 / tf32x3).
    The buffers start as all-ones bytes (NaN), so a field the export does not write cannot pass for a value."""
    import torch
    capi = _capi()
    prec, _ = capi.PRECISIONS[precision]
    engine.sets(beta, capi.UNSAFE_ANY)
    info = engine.pairs_prepare(capi.MODE_FANTASY, prec, beta)
    nx, rd, vb = info["n_x_local"], info["row_doubles"], info["vrow_bytes"]
    assert nx > 0, "no candidates: the case does not exercise the export"
    rows = torch.full((nx, rd), float("nan"), dtype=torch.float64, device="cuda")
    vrows = torch.full((nx, vb), 0xFF, dtype=torch.uint8, device="cuda")
    engine.pairs_export(rows, vrows)
    torch.cuda.synchronize()
    nc = engine.G - 1
    v = vrows.cpu().numpy().view(np.float64 if precision == "fp64" else np.uint32).reshape(nx, nc, -1)
    return rows.cpu().numpy(), v


def _check_exported(oracle, engine, ds, beta, kernel, P_grid, gidx, m, v, rows, V64):
    """Every field of the exported candidate rows [coords | ucb | xn | a | b | grid index] and the FP64 V rows against
    the oracle.  P_grid: all grid points; gidx: global index of each local point; m, v: the context's posterior."""
    d, G, n = P_grid.shape[1], m.shape[1], ds["X_norm"].shape[0]
    nc = G - 1
    lcb, ucb = oracle.bounds(m, v, beta)
    xs = np.flatnonzero(oracle.safe_mask(lcb))                   # local candidates, ascending
    assert rows.shape == (xs.size, 2 * d + 3 * nc + 1)
    assert np.array_equal(rows[:, -1], gidx[xs].astype(np.float64))
    coords = P_grid[gidx[xs]]
    assert np.array_equal(rows[:, :d], coords)                                               # numpy.linspace, bitwise
    assert np.array_equal(rows[:, d:d + nc], ucb[xs, 1:])                                    # FMA-free ucb, bitwise
    assert np.array_equal(rows[:, d + nc:2 * d + nc], (coords - ds["X_mean"]) / ds["X_std"])
    for c in range(nc):
        _, sf2, sn2 = oracle.unpack_hyper(ds["hypopt"][:, c + 1], d)
        vn = v[xs, c + 1] / ds["Y_std"][c + 1] ** 2
        den = vn + sn2 + oracle.EPS_F32
        np.testing.assert_allclose(rows[:, 2 * d + nc + c], beta * np.sqrt(vn) / den, rtol=AB_REL, atol=0)
        np.testing.assert_allclose(rows[:, 2 * d + 2 * nc + c], 1.0 / den, rtol=AB_REL, atol=0)
    # FP64 V rows: L_i^-1 k_i(X, x) of the oracle factor, exact zeros in the padding columns n .. npad-1
    assert V64.shape == (xs.size, nc, _npad(n))
    assert np.all(V64[:, :, n:] == 0.0)
    _, _, _, Vo = _reference(oracle, coords, ds, kernel, return_V=True)
    for c in range(nc):
        _, sf2, _ = oracle.unpack_hyper(ds["hypopt"][:, c + 1], d)
        err = np.max(np.abs(V64[:, c, :n] - Vo[c + 1]))
        assert err <= V_TOL * np.sqrt(sf2), (c, err)


def _check_tf32_rows(V64, V32, V3):
    """TF32 rows: cvt.rna.tf32.f32 of float32(FP64 row); split rows [hi | lo] with lo = tf32(float32(v - hi))."""
    npad = V64.shape[2]
    hi = round_tf32(V64.astype(np.float32))
    lo = round_tf32((V64 - hi.astype(np.float64)).astype(np.float32))
    assert V32.shape == V64.shape and V3.shape == (V64.shape[0], V64.shape[1], 2 * npad)
    assert np.array_equal(V32, hi.view(np.uint32))
    assert np.array_equal(V3[:, :, :npad], hi.view(np.uint32))
    assert np.array_equal(V3[:, :, npad:], lo.view(np.uint32))


def _cyclic_gidx(N, world, rank, block):
    """global indices of a rotated block-cyclic shard (common.cuh shard_global), as test_rotated_block_cyclic_shards."""
    nblk = (N + block - 1) // block
    sb = np.arange((nblk + world - 1) // world)
    gb = sb * world + (rank + sb + sb // world + sb // (world * world)) % world
    gb = gb[gb < nblk]
    return np.concatenate([np.arange(b * block, min(N, (b + 1) * block)) for b in gb])


# ---------------------------------------------------------------------------------------------------- 1. row blocks
def _full_grid_case(engine, oracle, name, n, kernel):
    ds, lo, hi, _ = _case(name, n)
    grid = GRIDS[name]
    engine.set_model(ds, kernel)
    engine.set_grid(lo, hi, grid)
    m, v = engine.posterior(with_grad=True)
    L = engine.lipschitz()
    P = oracle.make_grid(lo, hi, grid)
    fac, mo, vo = _reference(oracle, P, ds, kernel)
    em, ev = post_err(oracle, ds, m, v, mo, vo)
    assert em <= TOL_CHOL and ev <= TOL_CHOL, (em, ev)
    _check_lipschitz(L, P, ds, kernel, fac)


@pytest.mark.parametrize("n", N_LIST)
@pytest.mark.parametrize("name", ["c3", "d3", "d4"])
def test_posterior_across_row_blocks(engine, oracle, name, n):
    """npad = 128 ceil(n / 128): n just below, at and above the block edges 128 and 256 (1, 2 and 3 row blocks of the
    DMMA solve, its cross-block prefetch ring and its trimmed diagonal fragments)."""
    _full_grid_case(engine, oracle, name, n, "RBF")


@pytest.mark.parametrize("n", [2, 127, 128, 129, 257])
def test_matern52_posterior_across_row_blocks(engine, oracle, n):
    """The cross-covariance kernel is templated on the covariance function; the solve it feeds is not."""
    _full_grid_case(engine, oracle, "d4", n, "Matern52")


# ---------------------------------------------------------------------------------------------------- 2. chunks
@pytest.mark.parametrize("name,n", [("c3", 129), ("d4", 65)])
def test_chunked_posterior_is_the_one_chunk_posterior(engine, oracle, name, n):
    """posterior_chunk_mb = 1 raises the chunk to one wave of the solve (a few thousand points): the grid runs in
    several chunks and a ragged last one.  Per point the arithmetic is the one-chunk arithmetic, so mean, variance,
    Lipschitz constants and V rows are bitwise those of the one-chunk run -- and match the oracle."""
    ds, lo, hi, beta = _case(name, n)
    grid = BIG[name]
    N = int(np.prod(grid))
    assert N % 4 and N % 128
    engine.set_model(ds)
    engine.set_grid(lo, hi, grid)
    out = {}
    for mb in (1, 0):                     # chunked first: what the one-chunk run leaves in the buffers cannot help it
        with _options(engine, posterior_chunk_mb=mb):
            for kv, prec in ((1, "fp64"), (3, "tf32x3")):
                engine.kernel_launches(reset=True)
                m, v = engine.posterior(with_grad=True, keep_v=kv)
                launches = engine.kernel_launches(reset=True)
                L = engine.lipschitz()
                rows, V = _export(engine, beta, prec)
                out[mb, kv] = (m, v, L, rows, V, launches)
    for kv in (1, 3):
        a, b = out[1, kv], out[0, kv]
        assert a[5] >= 2 * b[5], ("expected several chunks", a[5], b[5])
        for x, y, what in zip(a[:5], b[:5], ("mean", "var", "lipschitz", "rows", "V rows")):
            assert np.array_equal(x, y), (kv, what)
    m, v, L, rows, V64, _ = out[1, 1]
    P = oracle.make_grid(lo, hi, grid)
    fac, mo, vo = _reference(oracle, P, ds, "RBF")
    em, ev = post_err(oracle, ds, m, v, mo, vo)
    assert em <= TOL_CHOL and ev <= TOL_CHOL, (em, ev)
    _check_lipschitz(L, P, ds, "RBF", fac)
    _check_exported(oracle, engine, ds, beta, "RBF", P, np.arange(N), m, v, rows, V64)


@pytest.mark.parametrize("name,n", [("c3", 129), ("d4", 65)])
def test_chunked_point_posterior_and_gradient(engine, oracle, name, n):
    """point_posterior / point_mean_grad over more explicit points than one chunk holds: bitwise the set_points +
    posterior() result on the same points (whose Lipschitz constant is max |grad|, bitwise), and the oracle's."""
    ds, lo, hi, _ = _case(name, n)
    d, G = ds["X_norm"].shape[1], ds["Y_norm"].shape[1]
    X = np.random.default_rng(17).uniform(lo, hi, size=(15013, d))
    engine.set_model(ds)
    g_one = [engine.point_mean_grad(X, i) for i in range(G)]
    with _options(engine, posterior_chunk_mb=1):
        engine.kernel_launches(reset=True)
        pm, pv = engine.point_posterior(X)
        launches = engine.kernel_launches(reset=True)
        g = [engine.point_mean_grad(X, i) for i in range(G)]
        engine.set_points(X)
        m, v = engine.posterior(with_grad=True)
        L = engine.lipschitz()
    assert launches >= 4, ("expected several chunks", launches)
    assert np.array_equal(pm, m) and np.array_equal(pv, v)
    fac, mo, vo = _reference(oracle, X, ds, "RBF")
    em, ev = post_err(oracle, ds, pm, pv, mo, vo)
    assert em <= TOL_CHOL and ev <= TOL_CHOL, (em, ev)
    for i in range(G):
        assert np.array_equal(g[i], g_one[i]), i
        assert np.max(np.abs(g[i])) == L[i], i
        go = R.mean_grad(X, ds, i, "RBF", factors=fac)
        assert np.max(np.abs(g[i] - go)) <= LIP_REL * np.max(np.abs(go)), i


# ---------------------------------------------------------------------------------------------------- 3. contiguous shards
CUTS = [7777, 15557, 23333]           # not multiples of 4, 32 or 128; the pieces hold 7777, 7780, 7776 and the rest


def _argbest(results, better):
    """reduce (index, value) pairs of the pieces like the device does: best value, lowest global index; -1 = empty"""
    best = (-1, None)
    for i, val in results:
        if i < 0:
            continue
        if best[0] < 0 or better(val, best[1]) or (val == best[1] and i < best[0]):
            best = (i, val)
    return best


@pytest.mark.parametrize("name,n", [("c3", 20), ("d3", 65)])
def test_contiguous_shards_are_slices_of_the_whole_grid(engine, oracle, name, n):
    """sbo_set_shard(first, count) pieces: posterior, sets masks, ball mask and Lipschitz constants are slices of the
    unsharded run, and the global indices the pieces report reduce to the unsharded sizes and arg-reductions."""
    capi = _capi()
    ds, lo, hi, beta = _case(name, n)
    grid = BIG[name]
    N = int(np.prod(grid))
    d = len(grid)
    cuts = [0] + CUTS + [N]
    counts = np.diff(cuts)
    assert (counts % 4 == 0).any() and (counts % 4 != 0).any()      # both the _v4 and the scalar set kernels run
    target = np.array([0.5 * (l + h) for l, h in zip(lo, hi)]) + 0.1 * (np.asarray(hi) - np.asarray(lo))
    x0, r = np.full(d, 0.3), 0.8
    kinds = (capi.ARGMAX_VAR0, capi.ARGMIN_LCB0, capi.ARGMIN_UCB0)
    MASKS = (capi.MASK_SAFE, capi.MASK_UNSAFE, capi.MASK_MIN)

    def run(min_ucb0=None):
        """posterior, sets (pass 2 against the GLOBAL min ucb_0, as a sharded step runs it), masks, arg-reductions"""
        m, v = engine.posterior(with_grad=True)
        L = engine.lipschitz()
        s1 = engine.sets_pass1(beta, capi.UNSAFE_ALL)
        s = engine.sets_pass2(s1["min_ucb0"] if min_ucb0 is None else min_ucb0)
        masks = [engine.mask(k) for k in MASKS]
        red = [engine.argreduce(k, capi.MASK_SAFE) for k in kinds]
        red.append(engine.argreduce(capi.ARGMIN_DIST, capi.MASK_SAFE, 0, target))
        ball = None
        if d == 3:
            engine.user_mask_ball(x0, r, capi.MASK_SAFE)
            ball = engine.mask(capi.MASK_USER)
        return m, v, L, s, masks, red, ball

    try:
        engine.set_model(ds)
        engine.set_grid(lo, hi, grid)
        m_f, v_f, L_f, s_f, masks_f, red_f, ball_f = run()
        pieces = []
        for a, b in zip(cuts[:-1], cuts[1:]):
            engine.set_shard(a, b - a)
            m, v, L, s, masks, red, ball = run(s_f["min_ucb0"])
            sl = slice(a, b)
            assert np.array_equal(m, m_f[sl]) and np.array_equal(v, v_f[sl]), a
            for k, got, want in zip(MASKS, masks, masks_f):
                assert np.array_equal(got, want[sl]), (a, k)
            if d == 3:
                assert np.array_equal(ball, ball_f[sl]), a
            with pytest.raises(ValueError):
                engine.stable_minmax(1)
            pieces.append((L, s, red))
        assert np.array_equal(np.max([p[0] for p in pieces], axis=0), L_f)
        for k in ("n_safe", "n_unsafe", "n_min"):
            assert sum(p[1][k] for p in pieces) == s_f[k], k
        for what, better in (("min_ucb0", lambda a, b: a < b), ("min_lcb0", lambda a, b: a < b), ("minimizer", lambda a, b: a > b)):
            iname, vname = (f"{what}_idx", what) if what != "minimizer" else ("minimizer_idx", "minimizer_var")
            got = _argbest([(p[1][iname], p[1][vname]) for p in pieces], better)
            assert got == (s_f[iname], s_f[vname]) or (got[0] < 0 and s_f[iname] < 0), what
        for j, better in enumerate([lambda a, b: a > b, lambda a, b: a < b, lambda a, b: a < b, lambda a, b: a < b]):
            got = _argbest([p[2][j] for p in pieces], better)
            assert got == red_f[j] or (got[0] < 0 and red_f[j][0] < 0), j
        assert s_f["n_safe"] > 0 and s_f["n_min"] > 0 and red_f[3][0] >= 0
        assert d != 3 or ball_f.any()
        # the oracle agrees with the unsharded run
        P = oracle.make_grid(lo, hi, grid)
        _, mo, vo = _reference(oracle, P, ds, "RBF")
        em, ev = post_err(oracle, ds, m_f, v_f, mo, vo)
        assert em <= TOL_CHOL and ev <= TOL_CHOL, (em, ev)
    finally:
        engine.set_grid(lo, hi, grid)


# ---------------------------------------------------------------------------------------------------- 4. V rows and exported rows
@pytest.mark.parametrize("layout", ["whole", "cyclic", "chunked"])
@pytest.mark.parametrize("name,n", [("c3", 20), ("d4", 129)])
def test_vrows_and_exported_rows(engine, oracle, name, n, layout):
    """posterior(keep_v = 1 | 2 | 3) -> sets -> pairs_prepare(FANTASY, fp64 | tf32 | tf32x3) -> pairs_export: the FP64 rows
    against the oracle's L^-1 k, the TF32 and split-TF32 rows bitwise against the TF32 rounding of the same context's
    FP64 rows, and every field of the candidate rows -- on the whole grid, one block-cyclic rank and in chunks."""
    capi = _capi()
    ds, lo, hi, beta = _case(name, n)
    grid = BIG[name] if name == "c3" else [9, 9, 9, 9]           # 31313 / 6561 points: several chunks at chunk_mb = 1
    N = int(np.prod(grid))
    engine.set_model(ds)
    engine.set_grid(lo, hi, grid)
    gidx = np.arange(N)
    if layout == "cyclic":
        gidx = _cyclic_gidx(N, 3, 1, 256)
        assert engine.set_shard_cyclic(1, 3, 256) == gidx.size
    res = {}
    try:
        with _options(engine, posterior_chunk_mb=1 if layout == "chunked" else DEFAULTS["posterior_chunk_mb"]):
            for precision in ("fp64", "tf32", "tf32x3"):
                engine.kernel_launches(reset=True)
                m, v = engine.posterior(keep_v=capi.PRECISIONS[precision][1])
                launches = engine.kernel_launches(reset=True)
                rows, V = _export(engine, beta, precision)
                res[precision] = (m, v, rows, V)
        if layout == "chunked":
            assert launches >= 4, ("expected several chunks", launches)
        m, v, rows, V64 = res["fp64"]
        for precision in ("tf32", "tf32x3"):
            assert np.array_equal(res[precision][0], m) and np.array_equal(res[precision][1], v), precision
            assert np.array_equal(res[precision][2], rows), precision
        P_grid = oracle.make_grid(lo, hi, grid)
        _, mo, vo = _reference(oracle, P_grid[gidx], ds, "RBF")
        em, ev = post_err(oracle, ds, m, v, mo, vo)
        assert em <= TOL_CHOL and ev <= TOL_CHOL, (em, ev)
        _check_exported(oracle, engine, ds, beta, "RBF", P_grid, gidx, m, v, rows, V64)
        _check_tf32_rows(V64, res["tf32"][3], res["tf32x3"][3])
    finally:
        engine.set_grid(lo, hi, grid)


# ---------------------------------------------------------------------------------------------------- 5. selectable paths
# The solve paths the posterior options select for an SE model on a meshgrid: the FP64 SIMT tiles (posterior_variant = 0),
# the cross-covariance from the separable factor tables (posterior_tables = 1) and the fused table solve
# (posterior_fused = 1).  Kept in a list of their own.
SELECTABLE = [{"posterior_variant": 0}, {"posterior_tables": 1}, {"posterior_fused": 1}]


@pytest.mark.parametrize("n", [65, 257])
@pytest.mark.parametrize("opts", SELECTABLE, ids=lambda o: "-".join(f"{k}={v}" for k, v in o.items()))
def test_selectable_posterior_paths_match_the_oracle(engine, oracle, opts, n):
    ds, lo, hi, beta = _case("d4", n)
    grid = GRIDS["d4"]
    engine.set_model(ds)
    engine.set_grid(lo, hi, grid)
    with _options(engine, **opts):
        m, v = engine.posterior(with_grad=True, keep_v=1)
        L = engine.lipschitz()
        rows, V64 = _export(engine, beta, "fp64")
    P = oracle.make_grid(lo, hi, grid)
    fac, mo, vo = _reference(oracle, P, ds, "RBF")
    em, ev = post_err(oracle, ds, m, v, mo, vo)
    assert em <= TOL_CHOL and ev <= TOL_CHOL, (em, ev)
    _check_lipschitz(L, P, ds, "RBF", fac)
    _check_exported(oracle, engine, ds, beta, "RBF", P, np.arange(P.shape[0]), m, v, rows, V64)
