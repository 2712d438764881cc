"""NumPy reference of the batch GoOSE acquisition (csrc/batch.cu, include/sbo_b200.h sbo_goose_batch), built on the FP64 oracle
and tests/safeopt_batch_ref.py (whose Downdate gives the objective variance given the data plus the pending picks).

Candidates C = S u T, raw units, lcb_0 = mean_0 - beta*sqrt(v) (the mean does not change).  Pick b, on v conditioned on the
earlier picks: S_b = S minus the earlier picks, T_b = T minus the targets earlier explore picks served; S_b empty: no pick;
(s, l_S) = argmin over S_b of lcb_0 and (t, l_T) over T_b (oracle.masked_argmin: lowest index on ties, (-1, +inf) if empty);
t = -1 or l_S <= l_T: the safe minimum s (test/test_GoOSE.py:158-162); else the point of S_b nearest to z_t
(oracle.explore_safeset restricted to S_b), and t is served.
"""
from __future__ import annotations

import numpy as np

import safeopt_batch_ref as SB
from oracle import gp_oracle as O


def pick_rule(points, lcb, S_b, T_b):
    """One pick on lcb_0 (N,) over boolean S_b / T_b: dict of the sbo_goose_batch_pick fields, or None if S_b is empty."""
    si, sl = O.masked_argmin(lcb, S_b)
    ti, tl = O.masked_argmin(lcb, T_b)
    if si < 0:
        return None
    p = {"idx": si, "explore": 0, "safe_lcb": sl, "safe_idx": si, "target_lcb": tl, "target_idx": ti, "dist": 0.0}
    if ti >= 0 and not sl <= tl:
        p["idx"], p["dist"] = O.explore_safeset(points, S_b, points[ti])
        p["explore"] = 1
    return p


def _top2_close(values, mask, best, tol):
    """Another member of the mask lies within tol of the best value."""
    if best < 0:
        return False
    rest = mask.copy()
    rest[best] = False
    return bool(rest.any()) and float(np.min(values[rest])) - values[best] <= tol


def near_tie(points, lcb, S_b, T_b, p, tol):
    """The pick is decided by values within tol (absolute, in lcb units): the top two of S_b or of T_b, l_S against l_T, or
    (explore) the two nearest points of S_b to the target (distances relative to the nearest one)."""
    if _top2_close(lcb, S_b, p["safe_idx"], tol) or _top2_close(lcb, T_b, p["target_idx"], tol):
        return True
    if p["target_idx"] >= 0 and abs(p["safe_lcb"] - p["target_lcb"]) <= tol:
        return True
    if p["explore"]:
        d2 = np.sum((points - points[p["target_idx"]]) ** 2, axis=1)
        return _top2_close(d2, S_b, p["idx"], 1e-9 * max(d2[p["idx"]], 1e-300))
    return False


def goose_batch(points, ds, mean0, var0, beta, S, T, q, kernel="RBF", forced=None, rtol=None, history=None):
    """The picks from the step's raw objective mean / variance (N,) and its S / T masks.  forced: (pick, served target or
    -1) per pick to condition on instead of the reference's own picks (to follow another implementation past a near tie).
    rtol: mark each pick with near_tie, at rtol times the largest |lcb_0| over C.  history: a list that receives
    (candidate indices, lcb_0 over them) before every pick.  Returns the list of pick dicts (min(q, |S|) of them)."""
    S, T = np.asarray(S, dtype=bool), np.asarray(T, dtype=bool)
    mean0 = np.asarray(mean0, dtype=np.float64)
    cand = np.flatnonzero(S | T)
    picks = []
    if cand.size == 0:
        return picks
    dd = SB.Downdate(points[cand], ds, np.asarray(var0)[cand], kernel)
    S_b, T_b = S.copy(), T.copy()
    lcb = np.full(S.shape[0], np.inf)
    for b in range(q):
        lcb[cand] = mean0[cand] - beta * np.sqrt(dd.v)
        if history is not None:
            history.append((cand, lcb[cand].copy()))
        p = pick_rule(points, lcb, S_b, T_b)
        if p is None:
            break
        if rtol is not None:
            p["near_tie"] = near_tie(points, lcb, S_b, T_b, p, rtol * float(np.max(np.abs(lcb[cand]))))
        picks.append(p)
        idx, served = forced[b] if forced is not None else (p["idx"], p["target_idx"] if p["explore"] else -1)
        S_b[idx] = False
        if served >= 0:
            T_b[served] = False
        if b + 1 < q:
            dd.commit(points[idx])
    return picks
