"""Drop-in mirror of the reference's ``models/SafeOpt.py`` (class ``BO``), restated on a dense grid.

The reference answers every question with a differential-evolution run over single-point jitted
inference (SafeOpt.py:47-124).  Here each acquisition step is ONE pass of the CUDA grid pipeline:
posterior over the grid -> lcb/ucb + packed safe / minimiser / unsafe bitmasks -> Lipschitz constant ->
expander pair kernel -> deterministic arg-reductions (lowest grid index on ties).  Same constructor
``BO(plant_system, bound, b)``, same methods and return values ``(x, value)``; results are grid points.

Additive keyword arguments (defaults reproduce the reference's semantics):
  grid_points_per_dim  400 for d <= 2 (the reference's plot grid, test/test_SafeOpt.py:325-326)
  expander_mode        'lipschitz' (reference-exact pair test) | 'fantasy' (north_star GEMM expander)
  precision            'fp64' | 'tf32' | 'tf32x3' (fantasy GEMM only; the tensor-core modes re-evaluate every pair inside their
                       error bound in FP64, so all three return the FP64 counts)
  unsafe_rule          'all' (reference: lcb_constraint_min returns the MAX, SafeOpt.py:73-77) | 'any'

Additive method ``Batch(q)``: q safe query points for parallel experiments from the same step (hallucinated variance
downdates of the objective GP; include/sbo_b200.h, sbo_safeopt_batch).
"""
from __future__ import annotations

import numpy as np

from .GP_Safe import GP
from ._boot import package


def default_grid_points(d):
    return 400 if d <= 2 else max(8, int(round(160000 ** (1.0 / d))))


class BO(GP):
    def __init__(self, plant_system, bound, b, grid_points_per_dim=None, expander_mode='lipschitz',
                 precision='fp64', unsafe_rule='all', device=0):
        GP.__init__(self, plant_system, device=device)
        self.bound = np.asarray(bound, dtype=np.float64)
        self.b = b
        self.GP_inference_jit = self.GP_inference
        self.grid_points_per_dim = grid_points_per_dim
        self.expander_mode = expander_mode
        self.precision = precision
        self.unsafe_rule = unsafe_rule
        self._grid_set = False
        self._step = None
        self._post_keep_v = None          # keep_v of the engine's last step posterior; None: the next step recomputes it

    # ------------------------------------------------------------------ grid pipeline plumbing
    def _capi(self):
        return package()._capi

    def _on_model_changed(self):
        self._step = None
        self._post_keep_v = None

    def _on_model_appended(self):
        # add_sample_fixed: the next step brings the last posterior up to the grown model (sbo_posterior_update)
        self._step = None

    def _ensure_grid(self):
        if not self._grid_set:
            d = self.bound.shape[0]
            pts = self.grid_points_per_dim
            if pts is None:
                pts = default_grid_points(d)
            pts = [int(pts)] * d if np.isscalar(pts) else [int(p) for p in pts]
            self.engine.set_grid(self.bound[:, 0], self.bound[:, 1], pts)
            self.grid_shape = tuple(pts)
            self._grid_set = True
            self._step = None
            self._post_keep_v = None

    def _ensure_step(self):
        """Posterior + sets for the current model, computed once per model version.  After add_sample_fixed the
        posterior is updated with the appended samples instead of recomputed."""
        self._ensure_uploaded(self.inference_datasets)
        self._ensure_grid()
        if self._step is None:
            capi = self._capi()
            fantasy = self.expander_mode == 'fantasy'
            keep_v = capi.PRECISIONS[self.precision][1] if fantasy else 0
            if self._post_keep_v == keep_v:
                self.engine.posterior_update(fetch=False)
            else:
                self.engine.posterior(with_grad=True, keep_v=keep_v, fetch=False)
                self._post_keep_v = keep_v
            rule = capi.UNSAFE_ALL if self.unsafe_rule == 'all' else capi.UNSAFE_ANY
            self._step = {"sets": self.engine.sets(self.b, rule), "L": self.engine.lipschitz()}
        return self._step

    def _x(self, idx):
        if idx < 0:
            return np.full(self.bound.shape[0], np.nan)
        return self.engine.point_coords(idx)

    def grid_posterior(self):
        """Additive: (mean (N,G), var (N,G)) over the grid (what vmap(GP_inference) returns)."""
        self._ensure_uploaded(self.inference_datasets)
        self._ensure_grid()
        self._step = None
        self._post_keep_v = None
        return self.engine.posterior(with_grad=False, keep_v=0, fetch=True)

    def safe_mask(self, kind='safe'):
        """Additive: bool mask over the grid ('safe' | 'minimizer' | 'unsafe' | 'expander')."""
        self._ensure_step()
        capi = self._capi()
        k = {'safe': capi.MASK_SAFE, 'minimizer': capi.MASK_MIN, 'unsafe': capi.MASK_UNSAFE,
             'expander': capi.MASK_EXPANDER}[kind]
        return self.engine.mask(k, 0)

    # ------------------------------------------------------------------ reference API
    def calculate_plant_outputs(self, x, noise=0):
        return np.array([plant(x, noise) for plant in self.plant_system])

    def mean(self, x, i):
        return self.GP_inference_jit(x, self.inference_datasets)[0][i]

    def ucb(self, x, i):
        m, v = self.GP_inference_jit(x, self.inference_datasets)
        return m[i] + self.b * np.sqrt(v[i])

    def lcb(self, x, i):
        m, v = self.GP_inference_jit(x, self.inference_datasets)
        return m[i] - self.b * np.sqrt(v[i])

    def lcb_constraint_min(self, x):
        """SafeOpt.py:73-77 -- returns the MAX of the constraint lcbs (sic)."""
        return max(self.lcb(x, i) for i in range(1, self.n_fun))

    def minimize_obj_ucb(self, safe_set_cons=None):
        """SafeOpt.py:47-51 -- min over the safe set of ucb_0 -> (x, value)."""
        s = self._ensure_step()["sets"]
        return self._x(s["min_ucb0_idx"]), s["min_ucb0"]

    def Minimizer(self):
        """SafeOpt.py:53-66 -- argmax var_0 over {x in S : lcb_0(x) <= min_S ucb_0} -> (x, std)."""
        s = self._ensure_step()["sets"]
        if s["minimizer_idx"] < 0:
            return self._x(-1), 0.0
        return self._x(s["minimizer_idx"]), float(np.sqrt(s["minimizer_var"]))

    def infnorm_mean_grad(self, x, i):
        """SafeOpt.py:68-71 -- || d mean_i / dx ||_inf at x (analytic gradient kernel)."""
        self._ensure_uploaded(self.inference_datasets)
        return float(np.max(np.abs(self.engine.point_mean_grad(x, i))))

    def maximize_infnorm_mean_grad(self, i):
        """SafeOpt.py:79-83 -- L_i = max over the grid of || grad mean_i ||_inf."""
        return float(self._ensure_step()["L"][i])

    def Lipschitz_continuity_constraint(self, x, i, max_infnorm_mean_grad):
        """SafeOpt.py:85-88 -- ucb_i(x) - L * ||x - z + 1e-8||, x = [x; z]."""
        d = self.nx_dim
        x = np.asarray(x, dtype=np.float64)
        return self.ucb(x[:d], i) - max_infnorm_mean_grad * np.linalg.norm(x[:d] - x[d:] + 1e-8)

    def Expander(self):
        """SafeOpt.py:90-124 -- most uncertain expander over all constraints -> (x, std)."""
        st = self._ensure_step()
        capi = self._capi()
        if "expander" not in st:
            if self.expander_mode == 'fantasy':
                prec = capi.PRECISIONS[self.precision][0]
                st["expander"] = self.engine.expander(self.b, None, capi.MODE_FANTASY, prec)
            else:
                L = np.full(self.n_fun, st["L"][self.n_fun - 1])   # SafeOpt.py:110: leaked i = n_fun-1
                st["expander"] = self.engine.expander(self.b, L, capi.MODE_LIPSCHITZ, capi.PREC_FP64)
        ex = st["expander"]
        if ex["best_idx"] < 0:
            return self._x(-1), 0.0
        return self._x(ex["best_idx"]), float(np.sqrt(ex["best_value"]))

    def Batch(self, q):
        """Additive: q safe query points of this step for parallel experiments -> (X (m, d), std (m,), info), m <= q.
        Pick 1 is the point the reference's decision rule takes (test/test_SafeOpt.py:153-158); each later pick applies the
        same rule to the objective variance conditioned on the earlier picks as pending observations (values unknown).  The
        safe, minimiser and expander sets stay those of the real data, so every point is in the safe set.  std[i] is the
        standard deviation of the set pick i was taken from; info["picks"] holds both sets' optima per pick.  m = 0 when the
        minimiser and expander sets are empty."""
        self.Expander()                     # the SafeOpt pair stage of the cached step (computed once per model version)
        picks = self.engine.safeopt_batch(q)
        d = self.bound.shape[0]
        X = np.array([self._x(p["idx"]) for p in picks], dtype=np.float64).reshape(len(picks), d)
        std = np.array([p["std_exp"] if p["from_expander"] else p["std_min"] for p in picks], dtype=np.float64)
        first = picks[0] if picks else {"std_min": 0.0, "std_exp": 0.0}
        info = {"picks": picks, "chose": ["expander" if p["from_expander"] else "minimizer" for p in picks],
                "std_minimizer": float(first["std_min"]), "std_expander": float(first["std_exp"])}
        return X, std, info
