"""CPU: the incremental grid posterior after appended samples (sbo_posterior_update), in NumPy against the FP64 oracle on the
grown data set, and the routing of the drivers and drop-in classes that use it.

Appending rows to the Cholesky factor leaves its leading block, and so the first n0 entries of v(p) = L^-1 k(X, p), unchanged;
with the rows r >= n0 of W' = L'^-1
    e_r(p) = sum_j W'[r][j] k_j(p),   var'(p) = max(0, var(p)/Y_std^2 - sum_r e_r(p)^2) Y_std^2,   V'(p) = [V(p) ; e(p)]."""
import numpy as np
import pytest
import scipy.linalg as sla

import matern_ref as R
from oracle import gp_oracle as O

TOL = 1e-12                       # |dvar| <= TOL * sf2 * Y_std^2 and |dV| <= TOL * sqrt(sf2), as the GPU comparisons


def _grown(d, n0, m, seed):
    """(ds0, ds1, P): a model with n0 samples, the same model with m more at the SAME normalisation (what
    sbo_append_sample holds), and grid points -- a box around the data plus every training point (var clamp case)."""
    rng = np.random.default_rng(seed)
    X = rng.uniform(-1.0, 1.0, size=(n0 + m, d))
    Y = np.column_stack([np.sin(X.sum(1)), 0.3 - 0.2 * (X ** 2).sum(1), np.cos(2 * X[:, 0])])
    hyp = np.vstack([rng.uniform(-0.5, 0.5, size=(d, 3)), rng.uniform(-0.2, 0.3, size=(1, 3)), np.full((1, 3), -3.5)])
    ds0 = O.make_inference_datasets(X[:n0], Y[:n0], hyp, with_inverse=False)
    ds1 = dict(ds0)
    ds1["X_norm"] = (X - ds0["X_mean"]) / ds0["X_std"]
    ds1["Y_norm"] = (Y - ds0["Y_mean"]) / ds0["Y_std"]
    P = np.vstack([rng.uniform(-1.2, 1.2, size=(300, d)), X])
    return ds0, ds1, P


def _update(P, ds0, ds1, var0, V0, kernel):
    """The update formula: (var', V' per GP) from the n0-sample posterior and the new rows of W'."""
    n0 = ds0["X_norm"].shape[0]
    d = P.shape[1]
    xn = (P - ds1["X_mean"]) / ds1["X_std"]
    var, V = np.empty_like(var0), []
    for i in range(ds1["Y_norm"].shape[1]):
        ell, sf2, _ = O.unpack_hyper(ds1["hypopt"][:, i], d)
        L = np.linalg.cholesky(R.build_K(ds1["X_norm"], ds1["hypopt"][:, i], kernel))
        Wn = sla.solve_triangular(L, np.eye(L.shape[0]), lower=True)[n0:]                 # the m new rows of W'
        e = Wn @ R.cov(ds1["X_norm"], xn, ell, sf2, kernel)                             # (m, N)
        y2 = ds1["Y_std"][i] ** 2
        var[:, i] = np.maximum(0.0, var0[:, i] / y2 - np.sum(e * e, axis=0)) * y2
        V.append(np.hstack([V0[i], e.T]))
    return var, V


@pytest.mark.parametrize("kernel", R.KERNELS)
@pytest.mark.parametrize("d,n0,m", [(2, 20, 1), (3, 40, 3), (4, 111, 17), (6, 120, 130)])
def test_update_formula_matches_the_grown_posterior(d, n0, m, kernel):
    ds0, ds1, P = _grown(d, n0, m, seed=100 * d + m)
    _, var0, V0 = R.posterior_chol(P, ds0, kernel, return_V=True)
    mean1, var1, V1 = R.posterior_chol(P, ds1, kernel, return_V=True)
    var, V = _update(P, ds0, ds1, var0, V0, kernel)
    for i in range(3):
        _, sf2, _ = O.unpack_hyper(ds1["hypopt"][:, i], d)
        scale = sf2 * ds1["Y_std"][i] ** 2
        assert np.max(np.abs(var[:, i] - var1[:, i])) <= TOL * scale, i
        assert np.max(np.abs(V[i] - V1[i])) <= TOL * np.sqrt(sf2), i
        assert np.array_equal(V[i][:, :n0], V0[i])                                       # old entries untouched
    # the training points (last n0 + m grid points): tiny variance, never negative; a clamped variance stays clamped
    assert np.all(var >= 0.0)
    clamped = var0 == 0.0
    assert np.all(var[clamped] == 0.0)


def test_update_formula_keeps_a_clamped_variance_at_zero():
    ds0, ds1, P = _grown(2, 12, 2, seed=5)
    _, var0, V0 = O.posterior_chol(P, ds0, return_V=True)
    var0[:4] = 0.0                                                                       # as if sf2 - |v|^2 <= 0 there
    var, _ = _update(P, ds0, ds1, var0, V0, "RBF")
    assert np.all(var[:4] == 0.0)


# ------------------------------------------------------------------------------------------------
# drivers: fixed_model=True appends with add_sample_fixed, the default keeps add_sample
# ------------------------------------------------------------------------------------------------
class _ScriptedBO:
    """Duck-typed BO with scripted answers that records how samples are added (as test_host_logic._ScriptedBO)."""
    nx_dim, n_fun = 2, 2

    def __init__(self, script):
        self.script, self.k, self.added = script, 0, []
        self.plant_system = [lambda x, noise=0: float(x[0] ** 2 + x[1] ** 2), lambda x, noise=0: float(1.0 - x[0])]

    def _cur(self):
        return self.script[min(self.k, len(self.script) - 1)]

    def Minimizer(self):
        return np.array(self._cur()["min"][0]), self._cur()["min"][1]

    def Expander(self):
        return np.array(self._cur()["exp"][0]), self._cur()["exp"][1]

    def minimize_obj_lcb(self):
        return np.array(self._cur()["safe"][0]), self._cur()["safe"][1]

    def Target(self):
        return np.array(self._cur()["tgt"][0]), self._cur()["tgt"][1]

    def explore_safeset(self, t):
        return np.asarray(t) * 0.5

    def calculate_plant_outputs(self, x, noise=0):
        return np.array([f(x, noise) for f in self.plant_system])

    def add_sample(self, x, y, hypopt=None):
        self.added.append(("add_sample", hypopt is not None))
        self.k += 1

    def add_sample_fixed(self, x, y):
        self.added.append(("add_sample_fixed", False))
        self.k += 1


SO_SCRIPT = [{"min": ([0.1, 0.2], 0.5), "exp": ([0.3, 0.4], 0.2)}, {"min": ([0.1, 0.2], 0.1), "exp": ([0.3, 0.4], 0.2)}]
GO_SCRIPT = [{"safe": ([0.2, 0.2], 0.10), "tgt": ([0.8, 0.8], 0.30)}, {"safe": ([0.2, 0.2], 0.50), "tgt": ([0.8, 0.4], 0.30)}]


@pytest.mark.parametrize("algo", ["safeopt", "goose"])
def test_drivers_route_appends_by_fixed_model(algo):
    from sbo_b200 import drivers

    def run(bo, **kw):
        if algo == "safeopt":
            return drivers.run_safeopt(bo, n_iteration=2, **kw)
        return drivers.run_goose(bo, n_iteration=2, f_opt=None, **kw)

    script = SO_SCRIPT if algo == "safeopt" else GO_SCRIPT
    runs = {}
    for kw, want in (({}, ("add_sample", False)), ({"hypopt": np.zeros((4, 2))}, ("add_sample", True)),
                     ({"fixed_model": True}, ("add_sample_fixed", False))):
        bo = _ScriptedBO(script)
        runs[want[0] + str(want[1])] = run(bo, **kw)
        assert bo.added == [want, want], kw
    # the decisions do not depend on how the samples were added
    ref = runs["add_sampleFalse"]
    for r in runs.values():
        assert [i["chose"] for i in r["info"]] == [i["chose"] for i in ref["info"]] and r["x_0"] == ref["x_0"]
    with pytest.raises(ValueError, match="fixed_model"):
        run(_ScriptedBO(script), fixed_model=True, hypopt=np.zeros((4, 2)))


# ------------------------------------------------------------------------------------------------
# SafeOpt.BO / GoOSE.BO: the step after add_sample_fixed updates the posterior, anything else recomputes it
# ------------------------------------------------------------------------------------------------
class _RecordingEngine:
    """Stands in for GridEngine: records the grid-posterior calls the drop-in classes make."""

    def __init__(self):
        self.calls = []

    def set_model(self, ds, kernel="RBF"):
        self.calls.append("set_model")

    def set_grid(self, lo, hi, pts):
        self.calls.append("set_grid")

    def append_sample(self, x, y):
        self.calls.append("append_sample")

    def posterior(self, with_grad=False, keep_v=0, fetch=True):
        self.calls.append(("posterior", bool(with_grad), int(keep_v)))

    def posterior_update(self, fetch=True):
        self.calls.append("posterior_update")
        return None, {"rows": 1, "recomputed": False}

    def sets(self, beta, rule):
        return {"min_lcb0_idx": 0, "min_lcb0": 0.0, "min_ucb0_idx": 0, "min_ucb0": 0.0, "minimizer_idx": -1, "minimizer_var": 0.0}

    def lipschitz(self):
        return np.ones(2)


@pytest.mark.parametrize("cls,mode", [("SafeOpt", "lipschitz"), ("SafeOpt", "fantasy"), ("GoOSE", "lipschitz"), ("GoOSE", "fantasy")])
def test_dropin_step_after_add_sample_fixed_uses_the_update(cls, mode):
    import importlib
    from sbo_b200 import _capi as capi
    from sbo_b200.problems import Benoit_Problem
    mod = importlib.import_module(f"sbo_b200.models.{cls}")
    bo = mod.BO([Benoit_Problem.Benoit_System_1, Benoit_Problem.con1_system_tight], [[-0.6, 1.5], [-1.0, 1.0]], 2.0,
                grid_points_per_dim=16, expander_mode=mode, precision="tf32")
    eng = _RecordingEngine()
    bo._engine = eng
    rng = np.random.default_rng(3)
    X = rng.uniform(-0.5, 0.5, size=(8, 2))
    Y = np.column_stack([[f(x) for x in X] for f in bo.plant_system])
    bo.GP_initialization(X, Y, 'RBF', multi_hyper=1, hypopt=np.tile([[0.1], [0.1], [0.2], [-3.0]], (1, 2)))
    kv = capi.PRECISIONS["tf32"][1] if mode == "fantasy" else 0
    full = ("posterior", True, kv)
    bo._ensure_step()
    assert eng.calls == ["set_model", "set_grid", full]
    for _ in range(2):                                       # step -> add_sample_fixed -> step: update, no upload
        eng.calls.clear()
        bo.add_sample_fixed([0.1, 0.1], [0.2, 0.3])
        bo._ensure_step()
        assert eng.calls == ["append_sample", "posterior_update"]
    eng.calls.clear()
    bo.grid_posterior()                                      # a posterior with other flags: the next step recomputes
    bo.add_sample_fixed([0.2, 0.1], [0.2, 0.3])
    bo._ensure_step()
    assert eng.calls == [("posterior", False, 0), "append_sample", full]
    eng.calls.clear()
    bo.set_hyperparameters(bo.hypopt)                        # a new model upload: the full path
    bo._ensure_step()
    assert eng.calls == ["set_model", full]
    eng.calls.clear()
    bo.expander_mode = "lipschitz" if mode == "fantasy" else "fantasy"    # other V rows wanted: recompute
    bo.add_sample_fixed([0.0, 0.1], [0.2, 0.3])
    bo._ensure_step()
    assert eng.calls == ["append_sample", ("posterior", True, 0 if mode == "fantasy" else capi.PRECISIONS["tf32"][1])]
