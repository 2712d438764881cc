"""Drop-in mirror of the reference's ``models/GoOSE.py`` (class ``BO``), restated on a dense grid.

``minimize_obj_lcb`` / ``Target`` / ``explore_safeset`` (GoOSE.py:63-119) each become one masked
arg-reduction (plus, for ``Target``, the pair kernel with the reduction over the safe side) of the CUDA
grid pipeline.  Same constructor and return values as the reference; ``expander_mode='fantasy'`` (with
``precision`` 'fp64' | 'tf32' | 'tf32x3') replaces the Lipschitz reachability test of ``Target`` by the
fantasy test of the SafeOpt expander: z is reachable if the GP update with y_i = ucb_i(x) makes it safe.

Additive method ``Batch(q)``: q distinct safe query points for parallel experiments from the same step (GoOSE's rule on
hallucinated variance downdates of the objective GP; include/sbo_b200.h, sbo_goose_batch).  It replaces the SafeOpt batch
that this class would otherwise inherit, which applies the SafeOpt rule to a GoOSE object.
"""
from __future__ import annotations

import numpy as np
from scipy.optimize import NonlinearConstraint

from .SafeOpt import BO as _GridBO


class BO(_GridBO):
    def __init__(self, plant_system, bound, b, grid_points_per_dim=None, unsafe_rule='all', device=0,
                 expander_mode='lipschitz', precision='fp64'):
        _GridBO.__init__(self, plant_system, bound, b, grid_points_per_dim=grid_points_per_dim,
                         expander_mode=expander_mode, precision=precision, unsafe_rule=unsafe_rule, device=device)
        # GoOSE.py:22-25 -- kept for API compatibility (SciPy constraint objects over lcb_i >= 0)
        self.safe_set_cons = [NonlinearConstraint(lambda x, i=i: self.lcb(x, i), 0., np.inf)
                              for i in range(1, self.n_fun)]

    def minimize_obj_lcb(self):
        """GoOSE.py:63-67 -- min over the safe set of lcb_0 -> (x, value)."""
        s = self._ensure_step()["sets"]
        return self._x(s["min_lcb0_idx"]), s["min_lcb0"]

    def Target(self):
        """GoOSE.py:80-114 -- lowest-lcb_0 unsafe point reachable from the safe set -> (z, lcb_0).
        Empty target set -> (nan, +inf) so the driver's ``min_safe_lcb <= target_lcb`` picks the safe minimiser."""
        st = self._ensure_step()
        if "target" not in st:
            capi = self._capi()
            if self.expander_mode == 'fantasy':
                st["target"] = self.engine.goose_target(self.b, None, capi.MODE_FANTASY, capi.PRECISIONS[self.precision][0])
            else:
                L = np.full(self.n_fun, st["L"][self.n_fun - 1])   # GoOSE.py:100: leaked i = n_fun-1
                st["target"] = self.engine.goose_target(self.b, L)
        tg = st["target"]
        if tg["best_idx"] < 0:
            return self._x(-1), np.inf
        return self._x(tg["best_idx"]), tg["best_value"]

    def explore_safeset(self, target):
        """GoOSE.py:116-119 -- the safe point nearest to ``target``."""
        self._ensure_step()
        capi = self._capi()
        idx, _ = self.engine.argreduce(capi.ARGMIN_DIST, capi.MASK_SAFE, 0, np.asarray(target, dtype=np.float64))
        return self._x(idx)

    def Batch(self, q):
        """Additive: q distinct safe query points of this step for parallel experiments -> (X (m, d), lcb (m,), info),
        m = min(q, number of safe grid points).  Pick 1 is the point the reference's decision rule takes
        (test/test_GoOSE.py:158-162); each later pick applies the same rule, over the safe points and targets not yet used,
        to lcb_0 with the objective variance conditioned on the earlier picks as pending observations (values unknown).
        The safe and target sets stay those of the real data, so every point is in the safe set.  lcb[i] is the lcb_0 of
        the set pick i was decided on (the safe minimum, or the target it explores towards); info holds the per-pick
        records ("picks"), "chose" ('safe_minimum' | 'explore'), "x_target" (m, d; NaN rows for safe picks) and pick 1's
        "min_safe_lcb" / "target_lcb"."""
        self.Target()                       # the GoOSE target stage of the cached step (computed once per model version)
        picks = self.engine.goose_batch(q)
        d = self.bound.shape[0]
        X = np.array([self._x(p["idx"]) for p in picks], dtype=np.float64).reshape(len(picks), d)
        lcb = np.array([p["target_lcb"] if p["explore"] else p["safe_lcb"] for p in picks], dtype=np.float64)
        x_target = np.array([self._x(p["target_idx"] if p["explore"] else -1) for p in picks], dtype=np.float64).reshape(len(picks), d)
        first = picks[0] if picks else {"safe_lcb": np.inf, "target_lcb": np.inf}
        info = {"picks": picks, "chose": ["explore" if p["explore"] else "safe_minimum" for p in picks], "x_target": x_target,
                "min_safe_lcb": float(first["safe_lcb"]), "target_lcb": float(first["target_lcb"])}
        return X, lcb, info
