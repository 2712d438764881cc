"""NumPy reference of the GP pipeline for any of the library's covariance functions ('RBF', 'Matern32', 'Matern52'), built on
the FP64 oracle (oracle/gp_oracle.py) and leaving it unchanged.

With s = sum_k (x_k - x'_k)^2 / ell_k (the oracle's direct-difference form):
    RBF       k = sf2 exp(-s/2)                     phi = k
    Matern32  k = sf2 (1 + t) exp(-t),  t = sqrt(3s)          phi = 3 sf2 exp(-t)
    Matern52  k = sf2 (1 + t + t^2/3) exp(-t),  t = sqrt(5s)  phi = (5/3) sf2 (1 + t) exp(-t)
with phi = -2 dk/ds, so that dk/dx_k = -phi (x_k - x'_k) / ell_k.  Everything else -- normalisation, prior mean, jitter,
bounds, sets, arg-reductions, the rank-1 fantasy update -- is the oracle's, so the 'RBF' branch reproduces it.
"""
from __future__ import annotations

import numpy as np
import scipy.linalg as sla

from oracle import gp_oracle as O

KERNELS = ("RBF", "Matern32", "Matern52")


def kval(s, sf2, kernel):
    if kernel == "RBF":
        return sf2 * np.exp(-0.5 * s)
    t = np.sqrt((3.0 if kernel == "Matern32" else 5.0) * np.maximum(s, 0.0))
    poly = 1.0 + t if kernel == "Matern32" else 1.0 + t + t * t / 3.0
    return sf2 * poly * np.exp(-t)


def phi(s, sf2, kernel):
    if kernel == "RBF":
        return kval(s, sf2, kernel)
    if kernel == "Matern32":
        return 3.0 * sf2 * np.exp(-np.sqrt(3.0 * np.maximum(s, 0.0)))
    t = np.sqrt(5.0 * np.maximum(s, 0.0))
    return (5.0 / 3.0) * sf2 * (1.0 + t) * np.exp(-t)


def cov(A, B, ell, sf2, kernel):
    """(|A|, |B|) covariance, direct differences."""
    return kval(O.sq_dist_direct(A, B, ell), sf2, kernel)


def build_K(X_norm, hyp_col, kernel):
    n, d = X_norm.shape
    ell, sf2, sn2 = O.unpack_hyper(hyp_col, d)
    return cov(X_norm, X_norm, ell, sf2, kernel) + (sn2 + O.EPS_F32) * np.eye(n)


def chol_factors(ds, kernel):
    G = ds["Y_norm"].shape[1]
    m0 = O.prior_mean(ds)
    out = []
    for i in range(G):
        L = np.linalg.cholesky(build_K(ds["X_norm"], ds["hypopt"][:, i], kernel))
        r = ds["Y_norm"][:, i] - m0[i]
        out.append((L, sla.solve_triangular(L.T, sla.solve_triangular(L, r, lower=True), lower=False)))
    return out


def posterior_chol(points, ds, kernel, block=16384, return_V=False, factors=None):
    """oracle.posterior_chol with the kernel `kernel`: (mean, var[, V rows]) in raw units."""
    points = np.atleast_2d(np.asarray(points, dtype=np.float64))
    N, d = points.shape
    G = ds["Y_norm"].shape[1]
    m0 = O.prior_mean(ds)
    fac = factors if factors is not None else chol_factors(ds, kernel)
    mean, var = np.empty((N, G)), np.empty((N, G))
    Vs = [np.empty((N, ds["X_norm"].shape[0])) for _ in range(G)] if return_V else None
    for s in range(0, N, block):
        xn = (points[s:s + block] - ds["X_mean"]) / ds["X_std"]
        for i in range(G):
            ell, sf2, _ = O.unpack_hyper(ds["hypopt"][:, i], d)
            L, alpha = fac[i]
            k = cov(ds["X_norm"], xn, ell, sf2, kernel)
            v = sla.solve_triangular(L, k, lower=True)
            mean[s:s + block, i] = (m0[i] + k.T @ alpha) * ds["Y_std"][i] + ds["Y_mean"][i]
            var[s:s + block, i] = np.maximum(0.0, sf2 - np.sum(v * v, axis=0)) * ds["Y_std"][i] ** 2
            if return_V:
                Vs[i][s:s + block] = v.T
    return (mean, var, Vs) if return_V else (mean, var)


def mean_grad(points, ds, i, kernel, block=32768, factors=None):
    """d mu_i / d x (raw units): (Ystd_i / Xstd_k) sum_j alpha_j (-phi_j (xn_k - Xn_jk) / ell_k)."""
    points = np.atleast_2d(np.asarray(points, dtype=np.float64))
    N, d = points.shape
    ell, sf2, _ = O.unpack_hyper(ds["hypopt"][:, i], d)
    a = (factors if factors is not None else chol_factors(ds, kernel))[i][1]
    Xn = ds["X_norm"]
    out = np.empty((N, d))
    for s in range(0, N, block):
        xn = (points[s:s + block] - ds["X_mean"]) / ds["X_std"]
        w = phi(O.sq_dist_direct(Xn, xn, ell), sf2, kernel) * a[:, None]
        for kk in range(d):
            diff = xn[None, :, kk] - Xn[:, None, kk]
            out[s:s + block, kk] = -(w * diff).sum(axis=0) / ell[kk] * ds["Y_std"][i] / ds["X_std"][kk]
    return out


def lipschitz_constant(points, ds, i, kernel, factors=None):
    return float(np.max(np.abs(mean_grad(points, ds, i, kernel, factors=factors))))


def negative_loglikelihood(hyper, X, Y, kernel):
    """oracle.negative_loglikelihood (GP_Safe.py:169-192) with the kernel `kernel`; Y is one (n, 1) column."""
    n, d = X.shape
    K = kval(O.sq_dist_direct(X, X, np.exp(2.0 * hyper[:d])), np.exp(2.0 * hyper[d]), kernel)
    K = K + (np.exp(2.0 * hyper[d + 1]) + 1e-8) * np.eye(n)
    L = np.linalg.cholesky((K + K.T) * 0.5)
    alpha = sla.solve_triangular(L.T, sla.solve_triangular(L, Y, lower=True), lower=False)
    return float(np.dot(Y.T, alpha)[0][0] + 2.0 * np.sum(np.log(np.diag(L))))


def fantasy_pairs(points, ds, beta, S, Z, kernel, block=256, dtype=np.float64, xs=None):
    """The fantasy pair decisions of oracle.fantasy_counts with the kernel `kernel`: -> (counts (N,), T (N,) bool).
    counts[x] = #z made safe by x (row sums), T = {z : some x makes z safe} (column OR).  `xs`: only these candidates
    (grid indices, a subset of S).  dtype="tf32" rounds the V operands to TF32 as the tensor-core emulation does."""
    N, d = points.shape
    G = ds["Y_norm"].shape[1]
    mu_n, var_n, Vs, xn = fantasy_terms(points, ds, kernel)
    xs = np.flatnonzero(S) if xs is None else np.asarray(xs)
    zs = np.flatnonzero(Z)
    counts, T = np.zeros(N, dtype=np.int64), np.zeros(N, dtype=bool)
    if xs.size == 0 or zs.size == 0:
        return counts, T
    hyp = ds["hypopt"]
    for s in range(0, xs.size, block):
        xb = xs[s:s + block]
        ok = np.ones((zs.size, xb.size), dtype=bool)
        for i in range(1, G):
            ell, sf2, sn2 = O.unpack_hyper(hyp[:, i], d)
            sn2 = sn2 + O.EPS_F32
            kzx = cov(xn[zs], xn[xb], ell, sf2, kernel)
            if dtype == "tf32":
                acc = O.round_tf32(Vs[i][zs]).astype(np.float64) @ O.round_tf32(Vs[i][xb]).astype(np.float64).T
            else:
                acc = Vs[i][zs] @ Vs[i][xb].T
            c = kzx - acc
            denom = var_n[xb, i] + sn2
            mu_p = mu_n[zs, i][:, None] + c * (beta * np.sqrt(var_n[xb, i]) / denom)[None, :]
            s2_p = var_n[zs, i][:, None] - c * c / denom[None, :]
            ok &= (mu_p - beta * np.sqrt(np.maximum(s2_p, 0.0))) >= 0.0
        counts[xb] = ok.sum(axis=0)
        T[zs] |= ok.any(axis=1)
    return counts, T


def fantasy_margin(points, ds, beta, S, Z, kernel, xs=None):
    """Per (z, x) pair min_i (mu' - beta sigma') in normalised units (|Z|, |xs|): finds pairs near the threshold."""
    N, d = points.shape
    G = ds["Y_norm"].shape[1]
    mu_n, var_n, Vs, xn = fantasy_terms(points, ds, kernel)
    xs = np.flatnonzero(S) if xs is None else np.asarray(xs)
    zs = np.flatnonzero(Z)
    out = np.full((zs.size, xs.size), np.inf)
    for i in range(1, G):
        ell, sf2, sn2 = O.unpack_hyper(ds["hypopt"][:, i], d)
        c = cov(xn[zs], xn[xs], ell, sf2, kernel) - Vs[i][zs] @ Vs[i][xs].T
        denom = var_n[xs, i] + sn2 + O.EPS_F32
        mu_p = mu_n[zs, i][:, None] + c * (beta * np.sqrt(var_n[xs, i]) / denom)[None, :]
        s2_p = var_n[zs, i][:, None] - c * c / denom[None, :]
        out = np.minimum(out, mu_p - beta * np.sqrt(np.maximum(s2_p, 0.0)))
    return out


def fantasy_terms(points, ds, kernel):
    """oracle.fantasy_terms with the kernel `kernel`: normalised mean and variance (N, G), V rows, normalised points."""
    mean, var, Vs = posterior_chol(points, ds, kernel, return_V=True)
    return mean / ds["Y_std"], var / ds["Y_std"] ** 2, Vs, (points - ds["X_mean"]) / ds["X_std"]


def fantasy_by_augmentation(x, zs, ds, beta, kernel):
    """oracle.fantasy_by_augmentation with the kernel `kernel`: add (x, ucb_i(x)) to every constraint GP at fixed
    normalisation and hyper-parameters and re-run the inverse-form inference at zs -> lcb' (|zs|, G) raw units."""
    x = np.asarray(x, dtype=np.float64).reshape(1, -1)
    zs = np.atleast_2d(zs)
    d, G = x.shape[1], ds["Y_norm"].shape[1]
    m0 = O.prior_mean(ds)
    mean_x, var_x = posterior_chol(x, ds, kernel)
    mz, vz = posterior_chol(zs, ds, kernel)
    out = np.empty((zs.shape[0], G))
    out[:, 0] = mz[:, 0] - beta * np.sqrt(vz[:, 0])
    xn, zn = (x - ds["X_mean"]) / ds["X_std"], (zs - ds["X_mean"]) / ds["X_std"]
    for i in range(1, G):
        ell, sf2, sn2 = O.unpack_hyper(ds["hypopt"][:, i], d)
        Xa = np.vstack([ds["X_norm"], xn])
        y_f = (mean_x[0, i] + beta * np.sqrt(var_x[0, i]) - ds["Y_mean"][i]) / ds["Y_std"][i]
        Ya = np.concatenate([ds["Y_norm"][:, i], [y_f]])
        iKa = np.linalg.inv(cov(Xa, Xa, ell, sf2, kernel) + (sn2 + O.EPS_F32) * np.eye(Xa.shape[0]))
        k = cov(Xa, zn, ell, sf2, kernel)
        mu = (m0[i] + k.T @ iKa @ (Ya - m0[i])) * ds["Y_std"][i] + ds["Y_mean"][i]
        s2 = np.maximum(0.0, sf2 - np.einsum("bn,nm,mb->b", k.T, iKa, k)) * ds["Y_std"][i] ** 2
        out[:, i] = mu - beta * np.sqrt(s2)
    return out


def safeopt_step(points, ds, beta, kernel, mode="lipschitz", unsafe_rule="all", L_override=None):
    """The SafeOpt decision (drivers.safeopt_iteration / test/test_SafeOpt.py:144-158) from the oracle's sets and
    arg-reductions on this kernel's posterior.  Lipschitz mode: L of constraint G-1 for every constraint (SafeOpt.py:110)."""
    G = ds["Y_norm"].shape[1]
    fac = chol_factors(ds, kernel)
    mean, var = posterior_chol(points, ds, kernel, factors=fac)
    lcb, ucb = O.bounds(mean, var, beta)
    S, Z = O.safe_mask(lcb), O.unsafe_mask(lcb, unsafe_rule)
    m_idx, m_std, M, min_ucb = O.minimizer(var, lcb, ucb, S)
    out = {"mean": mean, "var": var, "S": S, "Z": Z, "minimizer_idx": m_idx, "minimizer_std": m_std}
    if mode == "lipschitz":
        Ls = [0.0] + [lipschitz_constant(points, ds, i, kernel, fac) for i in range(1, G)] if L_override is None \
            else list(L_override)
        ex = O.expander_lipschitz(points, S, Z, ucb, var, [Ls[G - 1]] * G if L_override is None else Ls)
        out["L"] = Ls
        e_idx, e_std = ex["best_idx"], ex["best_std"]
        out["expander_mask"] = ex["masks"].any(axis=0)
    else:
        counts, _ = fantasy_pairs(points, ds, beta, S, Z, kernel)
        e_idx, v = O.masked_argmax(var[:, 0], counts > 0)
        e_std = float(np.sqrt(v)) if e_idx >= 0 else 0.0
        out["counts"] = counts
    out.update({"expander_idx": e_idx, "expander_std": e_std})
    out["x_new_idx"] = m_idx if m_std > e_std else e_idx
    return out


def goose_step(points, ds, beta, kernel, mode="lipschitz", unsafe_rule="all", L_override=None):
    """The GoOSE decision (drivers.goose_iteration / test/test_GoOSE.py:151-162) on this kernel's posterior."""
    G = ds["Y_norm"].shape[1]
    fac = chol_factors(ds, kernel)
    mean, var = posterior_chol(points, ds, kernel, factors=fac)
    lcb, ucb = O.bounds(mean, var, beta)
    S, Z = O.safe_mask(lcb), O.unsafe_mask(lcb, unsafe_rule)
    s_idx, s_lcb = O.minimize_obj_lcb(lcb, S)
    if mode == "lipschitz":
        Ls = [0.0] + [lipschitz_constant(points, ds, i, kernel, fac) for i in range(1, G)] if L_override is None \
            else list(L_override)
        tg = O.goose_target(points, S, Z, ucb, lcb, [Ls[G - 1]] * G if L_override is None else Ls)
        T = tg["masks"].any(axis=0)
        t_idx, t_lcb = tg["best_idx"], tg["best_lcb"]
    else:
        _, T = fantasy_pairs(points, ds, beta, S, Z, kernel)
        t_idx, t_lcb = O.masked_argmin(lcb[:, 0], T)
    out = {"mean": mean, "var": var, "S": S, "Z": Z, "T": T, "safe_min_idx": s_idx, "safe_min_lcb": s_lcb,
           "target_idx": t_idx, "target_lcb": t_lcb}
    if s_lcb <= t_lcb or t_idx < 0:
        out["x_new_idx"], out["explore_idx"] = s_idx, -1
    else:
        e_idx, _ = O.explore_safeset(points, S, points[t_idx])
        out["x_new_idx"] = out["explore_idx"] = e_idx
    return out


def fantasy_counts_at(xpts, zpts, ds, beta, kernel, block=8192):
    """Fantasy counts of the candidates xpts (raw coordinates) against the unsafe points zpts, with the V rows of the unsafe
    points computed block by block (full-size grids: the rows of every point would not fit the host)."""
    G, d = ds["Y_norm"].shape[1], xpts.shape[1]
    fac = chol_factors(ds, kernel)
    mx, vx, Vx = posterior_chol(xpts, ds, kernel, return_V=True, factors=fac)
    xn = (xpts - ds["X_mean"]) / ds["X_std"]
    counts = np.zeros(xpts.shape[0], dtype=np.int64)
    for s in range(0, zpts.shape[0], block):
        zb = zpts[s:s + block]
        mz, vz, Vz = posterior_chol(zb, ds, kernel, return_V=True, factors=fac)
        zn = (zb - ds["X_mean"]) / ds["X_std"]
        ok = np.ones((zb.shape[0], xpts.shape[0]), dtype=bool)
        for i in range(1, G):
            ell, sf2, sn2 = O.unpack_hyper(ds["hypopt"][:, i], d)
            ys2 = ds["Y_std"][i] ** 2
            c = cov(zn, xn, ell, sf2, kernel) - Vz[i] @ Vx[i].T
            denom = vx[:, i] / ys2 + sn2 + O.EPS_F32
            mu_p = (mz[:, i] / ds["Y_std"][i])[:, None] + c * (beta * np.sqrt(vx[:, i] / ys2) / denom)[None, :]
            s2_p = (vz[:, i] / ys2)[:, None] - c * c / denom[None, :]
            ok &= (mu_p - beta * np.sqrt(np.maximum(s2_p, 0.0))) >= 0.0
        counts += ok.sum(axis=0)
    return counts
