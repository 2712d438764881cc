"""CPU: the kernel-parametrised NumPy reference (tests/matern_ref.py) -- its SE branch against the pinned FP64 oracle, the
Matern kernels against their closed forms, central differences and brute-force augmented inference -- and the host GP's
Matern covariance and likelihood."""
import numpy as np
import pytest

import matern_ref as R

MATERN = ["Matern32", "Matern52"]


def _case(d=3, ppd=7, n=30, G=3, seed=11):
    from sbo_b200 import workloads
    ds, lo, hi, pts, beta = workloads.small(d=d, pts_per_dim=ppd, n=n, seed=seed, G=G)
    return ds, lo, hi, pts, beta


def test_se_branch_reproduces_the_oracle(oracle):
    ds, lo, hi, pts, beta = _case()
    P = oracle.make_grid(lo, hi, pts)
    m0, v0 = oracle.posterior_chol(P, ds)
    m1, v1 = R.posterior_chol(P, ds, "RBF")
    assert np.allclose(m1, m0, rtol=0, atol=1e-12 * np.abs(m0).max())
    assert np.allclose(v1, v0, rtol=0, atol=1e-12 * v0.max())
    dsi = oracle.make_inference_datasets(ds["X_norm"] * ds["X_std"] + ds["X_mean"], ds["Y_norm"] * ds["Y_std"] + ds["Y_mean"],
                                         ds["hypopt"])
    for i in range(ds["Y_norm"].shape[1]):
        g0, g1 = oracle.mean_grad(P, dsi, i), R.mean_grad(P, ds, i, "RBF")
        assert np.allclose(g1, g0, rtol=0, atol=1e-9 * np.abs(g0).max())
    h = ds["hypopt"][:, 1]
    y = ds["Y_norm"][:, 1:2]
    assert R.negative_loglikelihood(h, ds["X_norm"], y, "RBF") == pytest.approx(
        oracle.negative_loglikelihood(h, ds["X_norm"], y), rel=1e-12)
    lcb, _ = oracle.bounds(m0, v0, beta)
    S, Z = oracle.safe_mask(lcb), oracle.unsafe_mask(lcb, "any")
    assert S.any() and Z.any()
    counts, T = R.fantasy_pairs(P, ds, beta, S, Z, "RBF")
    assert np.array_equal(counts, oracle.fantasy_counts(P, ds, beta, S, Z))


@pytest.mark.parametrize("kernel", MATERN)
def test_matern_closed_forms_and_gradient(kernel):
    r = np.array([0.0, 0.1, 0.5, 1.0, 2.0, 4.0])
    sf2 = 1.7
    if kernel == "Matern32":
        want = sf2 * (1 + np.sqrt(3) * r) * np.exp(-np.sqrt(3) * r)
    else:
        want = sf2 * (1 + np.sqrt(5) * r + 5 * r * r / 3) * np.exp(-np.sqrt(5) * r)
    assert np.allclose(R.kval(r * r, sf2, kernel), want, rtol=1e-14, atol=0)
    s = np.linspace(0.01, 6.0, 50)
    h = 1e-6
    dk = (R.kval(s + h, sf2, kernel) - R.kval(s - h, sf2, kernel)) / (2 * h)
    assert np.allclose(R.phi(s, sf2, kernel), -2.0 * dk, rtol=1e-7, atol=1e-9)
    assert np.isfinite(R.phi(np.array([0.0]), sf2, kernel)).all()
    cK = 1.5 if kernel == "Matern32" else 5.0 / 6.0                       # |dk/ds| <= c_K sf2 (the FP32 error bound)
    assert np.max(np.abs(dk)) <= cK * sf2 * (1 + 1e-6)


@pytest.mark.parametrize("kernel", MATERN)
def test_mean_gradient_matches_central_differences(oracle, kernel):
    ds, lo, hi, pts, beta = _case()
    rng = np.random.default_rng(3)
    x = rng.uniform(-0.8, 0.8, size=(6, 3))
    h = 1e-6
    for i in range(ds["Y_norm"].shape[1]):
        g = R.mean_grad(x, ds, i, kernel)
        for k in range(3):
            e = np.zeros(3)
            e[k] = h
            fd = (R.posterior_chol(x + e, ds, kernel)[0][:, i] - R.posterior_chol(x - e, ds, kernel)[0][:, i]) / (2 * h)
            assert np.allclose(g[:, k], fd, rtol=1e-5, atol=1e-6 * np.abs(g).max())


@pytest.mark.parametrize("kernel", MATERN)
def test_rank1_fantasy_vs_augmented_inference(oracle, kernel):
    ds, lo, hi, pts, beta = _case(d=2, ppd=15, n=25)
    P = oracle.make_grid(lo, hi, pts)
    mean, var = R.posterior_chol(P, ds, kernel)
    lcb, _ = oracle.bounds(mean, var, beta)
    S, Z = oracle.safe_mask(lcb), oracle.unsafe_mask(lcb, "any")
    assert S.sum() >= 3 and Z.sum() >= 3
    margin = R.fantasy_margin(P, ds, beta, S, Z, kernel)
    xs, zs = np.flatnonzero(S), np.flatnonzero(Z)
    G = ds["Y_norm"].shape[1]
    for j in np.linspace(0, xs.size - 1, 4).astype(int):
        lcb_aug = R.fantasy_by_augmentation(P[xs[j]], P[zs], ds, beta, kernel)
        m_aug = (lcb_aug[:, 1:] / ds["Y_std"][1:]).min(axis=1)       # normalised units, min over the constraints
        assert np.allclose(margin[:, j], m_aug, rtol=1e-7, atol=1e-7)
    counts, T = R.fantasy_pairs(P, ds, beta, S, Z, kernel)
    assert np.array_equal(counts[xs], (margin >= 0).sum(axis=0))
    assert np.array_equal(T[zs], (margin >= 0).any(axis=1))


@pytest.mark.parametrize("kernel", MATERN)
def test_host_gp_matches_the_reference(kernel):
    from sbo_b200.models.GP_Safe import GP
    from sbo_b200.problems import Benoit_Problem as B
    gp = GP([B.Benoit_System_1, B.con1_system])
    ds, *_ = _case(d=2, n=20)
    X, Y = ds["X_norm"], ds["Y_norm"]
    gp.nx_dim = 2
    gp.kernel = kernel
    ell, sf2 = np.array([0.7, 1.3]), 1.4
    Kh = gp.Cov_mat(kernel, X, X, ell, sf2)
    assert np.allclose(Kh, R.cov(X, X, ell, sf2, kernel), rtol=0, atol=1e-12)
    hyp = np.array([0.1, -0.2, 0.3, -3.0])
    assert gp.negative_loglikelihood(hyp, X, Y[:, 1:2]) == pytest.approx(
        R.negative_loglikelihood(hyp, X, Y[:, 1:2], kernel), rel=1e-10)
    with pytest.raises(ValueError):
        gp.Cov_mat("Matern", X, X, ell, sf2)
