"""NumPy reference of the fantasy-mode GoOSE target, built on the FP64 oracle's fantasy primitives (oracle/gp_oracle.py).

For x in S and z in Z fantasise y_i = ucb_i(x) for every constraint GP i >= 1 and test lcb'_i(z | x) >= 0 (the quantities of
``fantasy_counts``).  The target set is T = {z in Z : some x in S makes z safe}: the column OR of the decisions whose row sums
are the expander counts.  The block loop below makes the same decisions as ``fantasy_counts`` (min over the constraints of
the margins is >= 0 exactly when every margin is) and also returns each z's best margin over x, in normalised units.
"""
from __future__ import annotations

import numpy as np

from oracle import gp_oracle as O


def fantasy_target_blocks(points, ds, beta, S, Z, block=256, dtype=np.float64):
    """-> (T, best): T bool (N,) the target set, best (N,) max over x in S of min_i margin'_i(z | x) (-inf outside Z).
    ``dtype="tf32"`` emulates the tensor-core operands as ``fantasy_counts`` does."""
    N, d = points.shape
    G = ds["Y_norm"].shape[1]
    mu_n, var_n, Vs, xn = O.fantasy_terms(points, ds, beta)
    xs, zs = np.flatnonzero(S), np.flatnonzero(Z)
    T = np.zeros(N, dtype=bool)
    best = np.full(N, -np.inf)
    if xs.size == 0 or zs.size == 0:
        return T, best
    hyp = ds["hypopt"]
    bz = np.full(zs.size, -np.inf)
    for s in range(0, xs.size, block):
        xb = xs[s:s + block]
        m = np.full((zs.size, xb.size), np.inf)
        for i in range(1, G):
            ell, sf2, sn2 = O.unpack_hyper(hyp[:, i], d)
            sn2 = sn2 + O.EPS_F32
            kzx = sf2 * np.exp(-0.5 * O.sq_dist_direct(xn[zs], xn[xb], ell))
            if dtype == "tf32":
                acc = O.round_tf32(Vs[i][zs]).astype(np.float64) @ O.round_tf32(Vs[i][xb]).astype(np.float64).T
            else:
                acc = (Vs[i][zs].astype(dtype) @ Vs[i][xb].astype(dtype).T).astype(np.float64)
            c = kzx - acc
            denom = var_n[xb, i] + sn2
            mu_p = mu_n[zs, i][:, None] + c * (beta * np.sqrt(var_n[xb, i]) / denom)[None, :]
            s2_p = var_n[zs, i][:, None] - c * c / denom[None, :]
            m = np.minimum(m, mu_p - beta * np.sqrt(np.maximum(s2_p, 0.0)))
        bz = np.maximum(bz, m.max(axis=1))
    T[zs] = bz >= 0.0
    best[zs] = bz
    return T, best


def goose_target_fantasy(points, ds, beta, S, Z, lcb, dtype=np.float64):
    """Fantasy GoOSE target: T, argmin lcb_0 over T (lowest index on ties; -1 / +inf when T is empty)."""
    T, best = fantasy_target_blocks(points, ds, beta, S, Z, dtype=dtype)
    i, v = O.masked_argmin(lcb[:, 0], T)
    return {"best_idx": i, "best_lcb": v, "mask": T, "best_margin": best}


def goose_step_fantasy(points, ds, beta, unsafe_rule="all"):
    """test/test_GoOSE.py:151-162 with the fantasy target (posterior in the Cholesky form the fantasy terms use)."""
    mean, var = O.posterior_chol(points, ds)
    lcb, ucb = O.bounds(mean, var, beta)
    S, Z = O.safe_mask(lcb), O.unsafe_mask(lcb, unsafe_rule)
    s_idx, s_lcb = O.minimize_obj_lcb(lcb, S)
    tg = goose_target_fantasy(points, ds, beta, S, Z, lcb)
    out = {"S": S, "Z": Z, "safe_min_idx": s_idx, "safe_min_lcb": s_lcb, "target_idx": tg["best_idx"],
           "target_lcb": tg["best_lcb"], "target_mask": tg["mask"], "best_margin": tg["best_margin"], "lcb": lcb}
    if s_lcb <= tg["best_lcb"] or tg["best_idx"] < 0:
        out["x_new_idx"], out["explore_idx"] = s_idx, -1
    else:
        e_idx, _ = O.explore_safeset(points, S, points[tg["best_idx"]])
        out["x_new_idx"] = out["explore_idx"] = e_idx
    return out
