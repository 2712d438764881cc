"""GPU: factorisation, NLL, grid posterior, appends and the fantasy pair stage at training sets up to the n the C ABI accepts
(sbo_set_model(_ex) and sbo_append_sample: n <= 16384; sbo_nll_batch(_ex): n <= 8192).

What depends on n here and runs nowhere else in the suite: the npad / 32 block steps of the Cholesky kernels and the
per-column-block walk of the triangular inverse, the one-CTA O(n^2) loops of k_alpha and k_append_row, the padding growth of
an append at npad = 16256 -> 16384, the > 48 KB shared-memory opt-in of k_nll_finish (npad >= 6144, i.e. n >= 6113), the
one-wave floor of the posterior chunk at large G npad, the npad / 128 row blocks of the DMMA solve, the V-row strides, the K
loop of the tensor-core fantasy GEMM and its K-dependent refinement band, and the FP64 row buffers of the refinement.

Data: workloads.synthetic (d = 3) with a distinct hyper-parameter per GP and dimension (test_gpu_hyper_layout.hyper_table,
with sn2 >= e^-6 so that cond(K) <= 1 + n sf2 / sn2 stays near 1e7 at n = 16384).  The training ball of radius 0.9 sits
inside a grid box of half-width 1, so that the safe set, the unsafe set, the fantasy expander and the refinement are all
non-empty; each test asserts that its stage did something.

Tolerances are exact or multiples of n u (u = 2^-53), each with its reason.  Where a constant c is not a textbook bound
(C_POST, C_MARGIN) it was set from the scatter between two FP64 routes (LAPACK Cholesky + triangular solves against the
explicit-inverse route this library takes) at n = 2049 and 4097 on these data sets, which stayed below c / 10.

Measured on one NVIDIA B200 (1000 W power limit): the module takes about 4 minutes, most of it the 128 appends at
n = 16256 .. 16384 and the host-side references; the n = 16384 fantasy case peaks at 57.7 GB of context memory."""
import functools

import numpy as np
import pytest
import scipy.linalg as sla
from scipy.linalg import lapack

import large_n_ref as LR
import matern_ref as R
from oracle import gp_oracle as O
from test_gpu_refine_cells import _forced

pytestmark = pytest.mark.gpu

U = LR.U
D = 3
SEED = 21
R_TRAIN, RADII, HALF_WIDTH = 0.9, (1.0, 1.1), 1.0
GRID = [29, 30, 28]                     # 24 360 points, a different count per axis
C_RES = 2.0     # Cholesky backward error: |L L^T - K| <= gamma_{n+1} |L||L^T| <= (n+1) u max K_ii, doubled for the blocked order
C_FWD = 4.0     # forward errors against LAPACK: c n u times the condition number each quantity carries (stated below)
C_POST = 4.0    # mean (relative to max(|mu|, Y_std)), var (in sf2 Y_std^2), V rows (in sqrt(sf2)), gradients: c n u
C_MARGIN = 64.0  # fantasy decisions: pairs within c n u sf2 (1 + gain) of the threshold may differ from the NumPy oracle


def _capi():
    from sbo_b200 import _capi
    return _capi


@pytest.fixture(scope="module")
def eng():
    """A context of its own: the n x n factors, V rows and pair buffers of this module (several GB) go with it."""
    import sbo_b200
    e = sbo_b200.GridEngine(0)
    yield e
    e.close()


def hyper_table(d, G, seed):
    """test_gpu_hyper_layout.hyper_table with 1/2 log sn2 over [-3, -2] (sn2 from e^-6 to e^-4)."""
    rng = np.random.default_rng(seed)
    hyp = np.empty((d + 2, G))
    hyp[:d] = rng.permutation(np.linspace(-0.7, 0.7, d * G)).reshape(d, G)
    hyp[d] = rng.permutation(np.linspace(-0.69, 0.69, G))
    hyp[d + 1] = rng.permutation(np.linspace(-3.0, -2.0, G))
    return hyp


@functools.lru_cache(maxsize=4)
def dataset(n, G):
    from sbo_b200 import workloads
    ds, _, _, _, beta = workloads.synthetic(D, 2, n, SEED, G, r_train=R_TRAIN, radii=RADII)
    ds["hypopt"] = hyper_table(D, G, SEED + G)
    return ds, beta


def _box():
    return np.full(D, 0.3 - HALF_WIDTH), np.full(D, 0.3 + HALF_WIDTH)


def _sf2(ds, i):
    return O.unpack_hyper(ds["hypopt"][:, i], D)[1]


def _get_factor(eng, which):
    """L (which = 0) or W (which = 1) of every GP through sbo_get_model, the other outputs NULL: (G, n, n) on the host."""
    out = np.empty((eng.G, eng.n, eng.n))
    p = _capi().dptr(out)
    eng._ck(eng._lib.sbo_get_model(eng._h, p if which == 0 else None, p if which == 1 else None, None))
    return out


# ---------------------------------------------------------------------------------------------------- 1. factorisation
@pytest.mark.parametrize("n,kernel", [(2049, "RBF"), (4097, "RBF"), (8192, "RBF"), (4097, "Matern52")])
def test_factorisation_against_numpy(eng, n, kernel):
    """L, W = L^-1 and alpha of sbo_set_model_ex against LAPACK's Cholesky, inverse and solves of the same K, and the residuals
    of the device factors themselves (products in FP64 by cuBLAS)."""
    import torch
    ds, _ = dataset(n, 2)
    eng.set_model(ds, kernel)
    L, W, alpha = eng.get_model()
    m0 = O.prior_mean(ds)
    for i in range(2):
        K = LR.model_K(ds, i, kernel)
        Lo = np.linalg.cholesky(K)
        Wo, info = lapack.dtrtri(Lo, lower=1)
        assert info == 0
        r = ds["Y_norm"][:, i] - m0[i]
        ao = sla.cho_solve((Lo, True), r)
        kap = LR.kappa_bound(ds, i)
        # residuals: Cholesky backward error (C_RES) and the triangular inverse, |W L - I| <= c n u |W||L|
        Lt, Wt, Kt = (torch.from_numpy(a).cuda() for a in (L[i], W[i], K))
        res = torch.max(torch.abs(Lt @ Lt.T - Kt)).item()
        assert res <= C_RES * n * U * np.max(np.diag(K)), (i, res / (n * U))
        resw = torch.max(torch.abs(Wt @ Lt - torch.eye(n, dtype=torch.float64, device="cuda"))).item()
        bw = torch.max(torch.abs(Wt) @ torch.abs(Lt)).item()
        assert resw <= C_RES * n * U * bw, (i, resw / (n * U * bw))
        # alpha = W^T (W r): k_alpha against the same products in cuBLAS order; each result is within 2 n u |W|^T (|W| |r|)
        # of the exact product (two nested n-term sums), so the two differ by at most twice that, elementwise
        rt = torch.from_numpy(r).cuda()
        at = torch.from_numpy(alpha[i]).cuda()
        a_blas = Wt.T @ (Wt @ rt)
        bound = 2 * C_RES * n * U * (torch.abs(Wt).T @ (torch.abs(Wt) @ torch.abs(rt)))
        assert bool(torch.all(torch.abs(at - a_blas) <= bound)), i
        del Lt, Wt, Kt
        # against LAPACK: two backward-stable factors of K differ by at most ~ kappa(L) n u |L| (kappa(L) = kappa(K)^1/2);
        # W = L^-1 and alpha = K^-1 r carry kappa(K) (k_alpha itself is pinned to the cuBLAS products above)
        sk = np.sqrt(kap)
        assert np.max(np.abs(L[i] - Lo)) <= C_FWD * n * U * sk * np.max(np.abs(Lo)), i
        assert np.max(np.abs(W[i] - Wo)) <= C_FWD * n * U * kap * np.max(np.abs(Wo)), i
        assert np.max(np.abs(alpha[i] - ao)) <= C_FWD * n * U * kap * np.max(np.abs(ao)), i
    torch.cuda.empty_cache()


def test_factorisation_at_the_limit(eng):
    """n = 16384 (npad = 16384, 512 block steps), G = 2: |L L^T - K| and |W L - I| in FP64 on the device, block by block,
    with K built by torch from the test's own data.  L and W come through sbo_get_model one at a time (2 GB per GP)."""
    import torch
    n = 16384
    ds, _ = dataset(n, 2)
    eng.set_model(ds)
    ref = LR.TorchSE(ds)
    del ref.L[:]                                    # only K is needed: keep the device footprint down
    L = _get_factor(eng, 0)
    Ls = [torch.from_numpy(L[i]).cuda() for i in range(2)]
    del L
    B = 2048
    for i in range(2):
        K = ref.K(i)
        kmax = torch.max(torch.diagonal(K)).item()
        res = max(torch.max(torch.abs(Ls[i][r:r + B] @ Ls[i].T - K[r:r + B])).item() for r in range(0, n, B))
        print(f"n = {n}, GP {i}: max |L L^T - K| = {res / (n * U * kmax):.3g} n u max K_ii")
        assert res <= C_RES * n * U * kmax, (i, res)
        del K
    W = _get_factor(eng, 1)
    for i in range(2):
        Wt = torch.from_numpy(W[i]).cuda()
        eye = torch.eye(n, dtype=torch.float64, device="cuda")
        res, bw = 0.0, 0.0
        for r in range(0, n, B):
            res = max(res, torch.max(torch.abs(Wt[r:r + B] @ Ls[i] - eye[r:r + B])).item())
            bw = max(bw, torch.max(torch.abs(Wt[r:r + B]) @ torch.abs(Ls[i])).item())
        print(f"n = {n}, GP {i}: max |W L - I| = {res / (n * U * bw):.3g} n u max |W||L|")
        assert res <= C_RES * n * U * bw, (i, res)
        del Wt, eye
    del W, Ls, ref
    torch.cuda.empty_cache()


def test_model_limit_is_refused_and_keeps_the_model(eng):
    """n = 16385 is SBO_ERR_INVALID; the installed model, its posterior and the call after it are unchanged."""
    ds, beta = dataset(2049, 3)
    big, _ = dataset(16385, 2)
    lo, hi = _box()
    eng.set_model(ds)
    eng.set_grid(lo, hi, GRID)
    m, v = eng.posterior()
    with pytest.raises(ValueError, match="n out of range"):
        eng.set_model(big)
    m2, v2 = eng.posterior()
    assert np.array_equal(m, m2) and np.array_equal(v, v2)
    assert eng.sets(beta, _capi().UNSAFE_ANY)["n_safe"] > 0


# ---------------------------------------------------------------------------------------------------- 2. NLL
@pytest.mark.parametrize("kernel", ["RBF", "Matern52"])
@pytest.mark.parametrize("n", [6112, 6113, 8192])
def test_nll_batch_across_the_shared_memory_opt_in(eng, n, kernel):
    """k_nll_finish keeps t[npad] in shared memory: 6112 is the last n within 48 KB (npad = 6112), 6113 the first beyond it
    (npad = 6144), 8192 the limit.  Three hyper-parameter rows, each with its own length-scales, sf2 and sn2."""
    ds, _ = dataset(n, 2)
    Xn, y = ds["X_norm"], ds["Y_norm"][:, 1]
    H = np.array([[-0.4, 0.1, 0.5, 0.3, -2.0], [0.2, -0.3, -0.1, -0.5, -2.6], [0.6, 0.4, -0.6, 0.0, -3.0]])
    got = eng.nll_batch(Xn, y, H, kernel)
    want = np.array([LR.nll(h, Xn, y, kernel) for h in H])
    assert np.unique(want).size == 3
    assert np.all(np.abs(got - want) <= 1e-9 * np.maximum(1.0, np.abs(want))), (got, want)


def test_nll_limit_is_refused(eng):
    ds, _ = dataset(8193, 2)
    H = np.array([[0.0, 0.0, 0.0, 0.0, -2.0]])
    with pytest.raises(ValueError, match="n out of range"):
        eng.nll_batch(ds["X_norm"], ds["Y_norm"][:, 1], H)
    ok = eng.nll_batch(ds["X_norm"][:8192], ds["Y_norm"][:8192, 1], H)
    assert np.isfinite(ok).all()


# ---------------------------------------------------------------------------------------------------- 3. grid posterior
def _export_dev(eng, beta):
    """sets -> pairs_prepare(FANTASY, fp64) -> pairs_export into torch CUDA tensors: (grid index of each candidate,
    V rows (n_x, G - 1, npad) float64), both on the device."""
    import torch
    capi = _capi()
    eng.sets(beta, capi.UNSAFE_ANY)
    info = eng.pairs_prepare(capi.MODE_FANTASY, capi.PREC_FP64, beta)
    nx, rd, vb = info["n_x_local"], info["row_doubles"], info["vrow_bytes"]
    assert nx > 0
    rows = torch.full((nx, rd), float("nan"), dtype=torch.float64, device="cuda")
    vrows = torch.full((nx, vb), 0xFF, dtype=torch.uint8, device="cuda")
    eng.pairs_export(rows, vrows)
    torch.cuda.synchronize()
    return rows[:, -1].to(torch.int64), vrows.view(torch.float64).reshape(nx, eng.G - 1, -1)


def _chunk_points(n, G, mb, count):
    """posterior.cu chunk_points: mb MB of Kx[G][npad][P], never below one wave of the solve (2 CTAs of 64 points per SM
    and GP), in multiples of 128 points."""
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    npad = -(-n // 128) * 128
    p = max((mb << 20) // (G * npad * 8), -(-2 * sms // G) * 64)
    return min(max(p // 128 * 128, 128), -(-count // 128) * 128)


def _posterior_run(eng, beta, chunk_mb):
    eng.set_option("posterior_chunk_mb", chunk_mb)
    try:
        eng.kernel_launches(reset=True)
        m, v = eng.posterior(with_grad=True, keep_v=1)
        launches = eng.kernel_launches(reset=True)
        Lip = eng.lipschitz()
        idx, V = _export_dev(eng, beta)
    finally:
        eng.set_option("posterior_chunk_mb", 0)
    return m, v, Lip, idx, V, launches


@pytest.mark.parametrize("n", [4097, 16384])
def test_grid_posterior_points_and_vrows(eng, n):
    """Grid mean / variance at 512 sampled points, every GP's Lipschitz constant over the whole grid, point_posterior and
    point_mean_grad at 64 points off the grid, and the FP64 V rows (keep_v = 1) of 64 sampled safe candidates, against the
    NumPy reference (n = 4097) or the torch FP64 reference (n = 16384).  The run in chunks of one solve wave
    (posterior_chunk_mb = 1) is bitwise the default one."""
    import torch
    ds, beta = dataset(n, 3)
    G = 3
    lo, hi = _box()
    eng.set_model(ds)
    eng.set_grid(lo, hi, GRID)
    P = O.make_grid(lo, hi, GRID)
    N = P.shape[0]
    one = _posterior_run(eng, beta, 0)
    cut = _posterior_run(eng, beta, 1)
    p_one, p_cut = _chunk_points(n, G, 1024, N), _chunk_points(n, G, 1, N)
    print(f"n = {n}: chunks of {p_one} / {p_cut} points, {one[5]} / {cut[5]} launches")
    assert -(-N // p_one) >= 2                          # the Kx tile of one wave is above 1 GiB at these n: several chunks
    assert p_cut == p_one or cut[5] > one[5], (p_cut, p_one, cut[5], one[5])
    for a, b, what in zip(one[:3], cut[:3], ("mean", "var", "lipschitz")):
        assert np.array_equal(a, b), what
    assert torch.equal(one[3], cut[3]) and torch.equal(one[4], cut[4]), "V rows"
    m, v, Lip, idx, V, _ = one
    del cut
    lcb, _ = O.bounds(m, v, beta)
    S, Z = O.safe_mask(lcb), O.unsafe_mask(lcb, "any")
    print(f"n = {n}: |S| = {S.sum()}, |Z| = {Z.sum()} of {N}")
    assert 0 < S.sum() < N and Z.sum() > 0
    rng = np.random.default_rng(n)
    samp = np.sort(rng.choice(N, 512, replace=False))
    X = rng.uniform(lo, hi, size=(64, D))
    cand = np.sort(rng.choice(idx.numel(), 64, replace=False))
    cidx = idx[cand].cpu().numpy()
    Vs = V[cand].cpu().numpy()
    pm, pv = eng.point_posterior(X)
    pg = [eng.point_mean_grad(X, i) for i in range(G)]
    if n <= 8192:
        fac = R.chol_factors(ds, "RBF")
        mo, vo = R.posterior_chol(P[samp], ds, "RBF", factors=fac)
        pmo, pvo = R.posterior_chol(X, ds, "RBF", factors=fac)
        _, _, Vo = R.posterior_chol(P[cidx], ds, "RBF", return_V=True, factors=fac)
        Lo = [np.max(np.abs(R.mean_grad(P, ds, i, "RBF", block=4096, factors=fac))) for i in range(G)]
        pgo = [R.mean_grad(X, ds, i, "RBF", factors=fac) for i in range(G)]
    else:
        ref = LR.TorchSE(ds)
        post = [ref.posterior(P[samp], i) for i in range(G)]
        mo, vo = np.column_stack([p[0] for p in post]), np.column_stack([p[1] for p in post])
        post = [ref.posterior(X, i) for i in range(G)]
        pmo, pvo = np.column_stack([p[0] for p in post]), np.column_stack([p[1] for p in post])
        Vo = [None] + [ref.posterior(P[cidx], i, return_V=True)[2] for i in range(1, G)]
        Lo = [np.max(np.abs(ref.mean_grad(P, i))) for i in range(G)]
        pgo = [ref.mean_grad(X, i) for i in range(G)]
        del ref
        torch.cuda.empty_cache()
    tol = C_POST * n * U
    for i in range(G):
        sf2, ys2 = _sf2(ds, i), ds["Y_std"][i] ** 2
        for got, want, what in ((m[samp], mo, "grid"), (pm, pmo, "points")):
            scale = max(np.max(np.abs(want[:, i])), ds["Y_std"][i])
            assert np.max(np.abs(got[:, i] - want[:, i])) <= tol * scale, (what, "mean", i)
        for got, want, what in ((v[samp], vo, "grid"), (pv, pvo, "points")):
            err = np.max(np.abs(got[:, i] - want[:, i]))
            print(f"n = {n}, GP {i} {what}: max |d var| = {err / (n * U * sf2 * ys2):.3g} n u sf2 Y_std^2")
            assert err <= tol * sf2 * ys2, (what, "var", i)
        assert abs(Lip[i] - Lo[i]) <= tol * Lo[i], ("lipschitz", i, Lip[i], Lo[i])
        assert np.max(np.abs(pg[i] - pgo[i])) <= tol * np.max(np.abs(pgo[i])), ("point_mean_grad", i)
        if i > 0:
            assert np.all(Vs[:, i - 1, n:] == 0.0)
            err = np.max(np.abs(Vs[:, i - 1, :n] - Vo[i]))
            assert err <= tol * np.sqrt(sf2), ("V rows", i, err / (n * U * np.sqrt(sf2)))
    del one, V, idx
    torch.cuda.empty_cache()


# ---------------------------------------------------------------------------------------------------- 4. appends
N0 = 16256                  # npad = 16256 = 127 x 128: the first append grows the padded factor to 16384


def _L_dev(eng):
    import torch
    L = _get_factor(eng, 0)
    out = torch.from_numpy(L).cuda()
    del L
    return out


def test_appends_across_the_padding_up_to_the_limit(eng):
    """16256 -> 16384 samples by 128 rank-1 appends (the first grows npad), G = 2: the appended factor against the one set
    from scratch (test_gpu_hyper_layout.test_model_factors_and_appends' tolerance, 1e-11 = 5.5 n u here), the incremental
    posterior without V rows against sbo_posterior on the appended model, a kept-V-row update across the padding growth
    that recomputes, and a 16385th append that is refused and leaves the model usable."""
    import torch
    n = 16384
    ds, beta = dataset(n, 2)
    ds0 = dict(ds, X_norm=ds["X_norm"][:N0], Y_norm=ds["Y_norm"][:N0])
    lo, hi = _box()
    eng.set_grid(lo, hi, GRID)
    # V rows kept (tf32): the first append changes the row stride, so the update runs the full posterior
    eng.set_model(ds0)
    eng.posterior(keep_v=2, fetch=False)
    eng.append_sample(ds["X_norm"][N0], ds["Y_norm"][N0])
    (mu1, vu1), info = eng.posterior_update()
    assert info == {"rows": 1, "recomputed": True}
    mf1, vf1 = eng.posterior(keep_v=2)
    assert np.array_equal(mu1, mf1) and np.array_equal(vu1, vf1)
    eng.release(3)
    # no V rows: the update is the m = 128 new rows of W
    eng.set_model(ds0)
    eng.posterior(fetch=False)
    for r in range(N0, n):
        eng.append_sample(ds["X_norm"][r], ds["Y_norm"][r])
    (mu, vu), info = eng.posterior_update()
    assert info == {"rows": n - N0, "recomputed": False}
    mf, vf = eng.posterior()
    assert np.array_equal(mu, mf)
    for i in range(2):
        sf2, ys2 = _sf2(ds, i), ds["Y_std"][i] ** 2
        err = np.max(np.abs(vu[:, i] - vf[:, i]))
        assert err <= C_POST * n * U * sf2 * ys2, (i, err / (n * U * sf2 * ys2))
    La = _L_dev(eng)
    # the 16385th append: refused, nothing changed
    with pytest.raises(ValueError, match="n out of range"):
        eng.append_sample(np.zeros(D), np.zeros(2))
    assert eng.n == n
    m2, v2 = eng.posterior()
    assert np.array_equal(m2, mf) and np.array_equal(v2, vf)
    eng.set_model(ds)
    Lb = _L_dev(eng)
    err = torch.max(torch.abs(La - Lb)).item()
    scale = torch.max(torch.abs(Lb)).item()
    print(f"appended vs from-scratch L at n = {n}: {err / (n * U * scale):.3g} n u max |L|")
    assert err <= 1e-11 * scale
    del La, Lb
    torch.cuda.empty_cache()


# ---------------------------------------------------------------------------------------------------- 5. fantasy pair stage
def _fantasy(eng, beta, precision, goose=False):
    capi = _capi()
    prec, keep_v = capi.PRECISIONS[precision]
    eng.posterior(keep_v=keep_v, fetch=False)
    s = eng.sets(beta, capi.UNSAFE_ANY)
    if goose:
        tg = eng.goose_target(beta, None, capi.MODE_FANTASY, prec)
        return s, tg, eng.mask(capi.MASK_TARGET, 0)
    ex = eng.expander(beta, None, capi.MODE_FANTASY, prec, want_counts=True)
    return s, ex, eng.refine_stats()


@pytest.mark.parametrize("n", [4097, 16384])
def test_fantasy_expander_refined_counts_are_the_fp64_counts(eng, n):
    """G = 3, d = 3, 24 360 grid points.  The refined tf32 and tf32x3 counts (fantasy_refine = 2) are identical to the FP64
    mode's (k_fantasy_dmma), with the same expander set and best index; bounds mode brackets the FP64 set; a refinement cut
    into cells by a small fantasy_refine_mb gives the same counts.  At n = 4097 the FP64 counts of 32 sampled candidates
    against every unsafe point match the NumPy oracle up to pairs within C_MARGIN n u sf2 (1 + gain) of the threshold."""
    capi = _capi()
    ds, beta = dataset(n, 3)
    lo, hi = _box()
    eng.set_model(ds)
    eng.set_grid(lo, hi, GRID)
    N = int(np.prod(GRID))
    try:
        s, ex64, st64 = _fantasy(eng, beta, "fp64")
        c64 = ex64["counts"]
        print(f"n = {n} fp64: |S| {s['n_safe']}, |Z| {s['n_unsafe']}, expanders {int((c64 > 0).sum())}, best {ex64['best_idx']}")
        assert 0 < s["n_safe"] < N and s["n_unsafe"] > 0, s
        assert (c64 > 0).any(), "no fantasy expander"
        for precision in ("tf32", "tf32x3"):
            _, ex, st = _fantasy(eng, beta, precision)
            print(f"n = {n} {precision}: n_ambiguous {ex['n_ambiguous']}, n_refined_safe {ex['n_refined_safe']}, "
                  f"refine_stats {st}, mem peak {eng.mem_peak() / 2 ** 30:.2f} GB")
            assert ex["n_ambiguous"] > 0 and st["cells"] >= 1 and st["fp64_rows"] > 0, (precision, ex["n_ambiguous"], st)
            d = ex["counts"] != c64
            assert not d.any(), (precision, int(d.sum()), np.flatnonzero(d)[:8])
            assert ex["best_idx"] == ex64["best_idx"] and ex["n_hit"] == ex64["n_hit"], precision
            if precision == "tf32":
                def run():
                    return eng.expander(beta, None, capi.MODE_FANTASY, capi.PREC_TF32, want_counts=True)
                mb, cutr, stc = _forced(eng, run, ex, st, min_cells=2)
                print(f"n = {n} tf32 in cells: {mb} MB, refine_stats {stc}")
                assert stc["cells"] >= 2, stc
                assert np.array_equal(cutr["counts"], c64) and cutr["best_idx"] == ex64["best_idx"]
        try:
            eng.set_option("fantasy_refine", 3)
            _, bd, _ = _fantasy(eng, beta, "tf32")
        finally:
            eng.set_option("fantasy_refine", 2)
        cb, und = bd["counts"], bd["counts"] < 0
        print(f"n = {n} bounds mode: certified {int((cb > 0).sum())}, undecided {int(und.sum())}")
        assert (cb > 0).any()
        assert np.all(cb[~und] <= c64[~und])
        assert np.all(c64[cb > 0] > 0) and np.all((cb > 0) | und | (c64 == 0))
        if n <= 8192:
            _fp64_against_the_oracle(eng, ds, beta, c64)
    finally:
        eng.release(3)


def _fp64_against_the_oracle(eng, ds, beta, c64):
    """32 candidates (30 evenly spaced over S, and the largest and smallest constraint-1 variance) against all of Z."""
    lo, hi = _box()
    P = O.make_grid(lo, hi, GRID)
    n = ds["X_norm"].shape[0]
    m, v = eng.posterior()
    lcb, _ = O.bounds(m, v, beta)
    S, Z = O.safe_mask(lcb), O.unsafe_mask(lcb, "any")
    xs = np.flatnonzero(S)
    pick = np.unique(np.concatenate([xs[np.linspace(0, xs.size - 1, 30).astype(int)],
                                     [xs[np.argmax(v[xs, 1])], xs[np.argmin(v[xs, 1])]]]))
    fac = R.chol_factors(ds, "RBF")
    marg = LR.fantasy_margins(P[pick], P[Z], ds, beta, "RBF", fac)
    want = (marg >= 0.0).sum(axis=0)
    gain, sf2max = np.zeros(pick.size), 0.0
    for i in range(1, 3):
        _, sf2, sn2 = O.unpack_hyper(ds["hypopt"][:, i], D)
        sf2max = max(sf2max, sf2)
        vn = v[pick, i] / ds["Y_std"][i] ** 2
        gain = np.maximum(gain, beta * np.sqrt(vn) / (vn + sn2 + O.EPS_F32))
    near = (np.abs(marg) <= C_MARGIN * n * U * sf2max * (1.0 + gain)[None, :]).sum(axis=0)
    dc = np.abs(c64[pick].astype(np.int64) - want)
    print(f"n = {n} fp64 vs oracle: {pick.size} candidates x {int(Z.sum())} z, {int(want.sum())} newly-safe pairs, "
          f"{int((dc > 0).sum())} differ, near-threshold pairs {int(near.sum())}")
    assert want.sum() > 0
    assert np.all(dc <= near), (pick[dc > near], dc[dc > near], near[dc > near])


def test_fantasy_goose_target_at_the_limit(eng):
    """n = 16384, tf32: the fantasy GoOSE target mask and its arg-min lcb_0 are those of the FP64 mode."""
    n = 16384
    ds, beta = dataset(n, 3)
    lo, hi = _box()
    eng.set_model(ds)
    eng.set_grid(lo, hi, GRID)
    try:
        _, t64, T64 = _fantasy(eng, beta, "fp64", goose=True)
        _, t32, T32 = _fantasy(eng, beta, "tf32", goose=True)
        print(f"n = {n} GoOSE target: |T| {int(T64.sum())}, best {t64['best_idx']}, tf32 n_ambiguous {t32['n_ambiguous']}, "
              f"mem peak {eng.mem_peak() / 2 ** 30:.2f} GB")
        assert T64.any()
        assert np.array_equal(T32, T64) and t32["best_idx"] == t64["best_idx"] and t32["best_value"] == t64["best_value"]
    finally:
        eng.release(3)
