"""NumPy reference of the batch SafeOpt acquisition (csrc/batch.cu, include/sbo_b200.h sbo_safeopt_batch), built on the FP64
oracle and tests/matern_ref.py (the 'RBF' branch there reproduces the oracle).

Objective GP (index 0), normalised units, noise of a hallucinated observation sn = exp(2 hyp[d+1, 0]) + eps_f32:
  * brute force: append the normalised picks to X_norm (any Y) and rerun the Cholesky posterior -- the exact posterior
    variance given the n observations plus the pending ones;
  * incremental: c(p, x) = k(p, x) - k(X, p)^T K^-1 k(X, x), [c(x_i, x_j)] + sn I = R R^T grown one row per pick,
    w_b(p) = (c(p, x_b) - sum_{j<b} R_bj w_j(p)) / R_bb, v_b(p) = max(0, v_{b-1}(p) - w_b(p)^2)  (the kernels' formula).
The pick rule (test/test_SafeOpt.py:153-158 with drivers.safeopt_iteration's fallback) acts on boolean M / E masks and raw
variances: std = sqrt(max over the set of v * Y_std0^2), lowest index on ties; M's point if std_M > std_E, else E's; an empty
set yields to the other; both empty: no pick.
"""
from __future__ import annotations

import numpy as np
import scipy.linalg as sla

import matern_ref as MR
from oracle import gp_oracle as O


def objective_factor(ds, kernel):
    """(ell, sf2, sn, L) of GP 0: K = L L^T with the model's diagonal sn2 + eps_f32 (GP_Safe.py:229-231)."""
    d = ds["X_norm"].shape[1]
    ell, sf2, sn2 = O.unpack_hyper(ds["hypopt"][:, 0], d)
    L = np.linalg.cholesky(MR.build_K(ds["X_norm"], ds["hypopt"][:, 0], kernel))
    return ell, sf2, sn2 + O.EPS_F32, L


def variance_bruteforce(points, ds, pick_points, kernel="RBF"):
    """Raw objective variance over `points` given the data plus observations at `pick_points` (values irrelevant)."""
    pick_points = np.atleast_2d(np.asarray(pick_points, dtype=np.float64))
    aug = dict(ds)
    aug["X_norm"] = np.vstack([ds["X_norm"], (pick_points - ds["X_mean"]) / ds["X_std"]])
    aug["Y_norm"] = np.vstack([ds["Y_norm"], np.zeros((pick_points.shape[0], ds["Y_norm"].shape[1]))])
    return MR.posterior_chol(points, aug, kernel)[1][:, 0]


class Downdate:
    """Incremental objective variance over the candidate points `cand_points`, starting from their raw variances var0."""

    def __init__(self, cand_points, ds, var0, kernel="RBF", block=8192):
        self.ds, self.kernel = ds, kernel
        self.ell, self.sf2, self.sn, self.L = objective_factor(ds, kernel)
        self.xn = (np.asarray(cand_points, dtype=np.float64) - ds["X_mean"]) / ds["X_std"]
        self.Kxc = np.empty((ds["X_norm"].shape[0], self.xn.shape[0]))
        for s in range(0, self.xn.shape[0], block):
            self.Kxc[:, s:s + block] = MR.cov(ds["X_norm"], self.xn[s:s + block], self.ell, self.sf2, kernel)
        self.v = np.asarray(var0, dtype=np.float64).copy()
        self.ys2 = float(ds["Y_std"][0]) ** 2
        self.xb, self.kb, self.ub, self.R, self.w = [], [], [], [], []

    def _k(self, A, B):
        return MR.cov(np.atleast_2d(A), np.atleast_2d(B), self.ell, self.sf2, self.kernel)

    def commit(self, x_raw):
        """Hallucinate an observation at raw point x_raw: v <- v - w^2 * Y_std0^2 (clamped at 0)."""
        xb = (np.asarray(x_raw, dtype=np.float64) - self.ds["X_mean"]) / self.ds["X_std"]
        kb = self._k(self.ds["X_norm"], xb)[:, 0]
        ub = sla.cho_solve((self.L, True), kb)
        b = len(self.xb)
        a = np.array([self._k(xb, self.xb[j])[0, 0] - kb @ self.ub[j] for j in range(b)] + [self.sf2 - kb @ ub + self.sn])
        r = np.zeros(b + 1)
        for j in range(b):
            r[j] = (a[j] - r[:j] @ self.R[j][:j]) / self.R[j][j]
        r[b] = np.sqrt(max(a[b] - r[:b] @ r[:b], self.sn))
        c = self._k(self.xn, xb)[:, 0] - self.Kxc.T @ ub
        wb = (c - sum(r[j] * self.w[j] for j in range(b))) / r[b]
        self.v = np.maximum(0.0, self.v - wb * wb * self.ys2)
        self.xb.append(xb); self.kb.append(kb); self.ub.append(ub); self.R.append(r); self.w.append(wb)


def pick_rule(v, M, E):
    """One pick on raw variances v (N,) over boolean masks: dict of the sbo_batch_pick fields, or None if M and E are empty."""
    im, vm = O.masked_argmax(v, M)
    ie, ve = O.masked_argmax(v, E)
    if im < 0 and ie < 0:
        return None
    sm = float(np.sqrt(vm)) if im >= 0 else 0.0
    se = float(np.sqrt(ve)) if ie >= 0 else 0.0
    take_min = im >= 0 and (ie < 0 or sm > se)
    return {"idx": im if take_min else ie, "from_expander": 0 if take_min else 1, "std_min": sm, "idx_min": im,
            "std_exp": se, "idx_exp": ie}


def _near_tie(v, mask, best, rtol):
    """The best std of the set and the next best (another index) lie within rtol of each other."""
    if best < 0:
        return False
    rest = mask.copy()
    rest[best] = False
    if not rest.any():
        return False
    s1, s2 = np.sqrt(v[best]), np.sqrt(np.max(v[rest]))
    return s1 - s2 <= rtol * max(s1, 1e-300)


def near_tie(v, M, E, pick, rtol):
    """The pick is decided by values within rtol: the top two of M or of E, or std_M against std_E of two different points
    (one point best in both sets, M and E overlap, gives equal stds and an exact decision)."""
    if _near_tie(v, M, pick["idx_min"], rtol) or _near_tie(v, E, pick["idx_exp"], rtol):
        return True
    sm, se = pick["std_min"], pick["std_exp"]
    return (pick["idx_min"] >= 0 and pick["idx_exp"] >= 0 and pick["idx_min"] != pick["idx_exp"]
            and abs(sm - se) <= rtol * max(sm, se, 1e-300))


def safeopt_batch(points, ds, var0, M, E, q, kernel="RBF", forced=None, rtol=None):
    """The q picks from the step's raw objective variance var0 (N,) and its M / E masks.  forced: global indices to
    condition on instead of the reference's own picks (to follow another implementation past a near tie).  rtol: mark
    each pick with near_tie.  Returns the list of pick dicts (shorter than q only when M and E are empty)."""
    M, E = np.asarray(M, dtype=bool), np.asarray(E, dtype=bool)
    cand = np.flatnonzero(M | E)
    dd = Downdate(points[cand], ds, np.asarray(var0)[cand], kernel)
    v = np.zeros(M.shape[0])
    picks = []
    for b in range(q):
        v[cand] = dd.v
        p = pick_rule(v, M, E)
        if p is None:
            break
        if rtol is not None:
            p["near_tie"] = near_tie(v, M, E, p, rtol)
        picks.append(p)
        if b + 1 < q:
            dd.commit(points[forced[b] if forced is not None else p["idx"]])
    return picks
