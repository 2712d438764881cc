"""Drop-in mirror of the reference's ``models/GP_Safe.py`` (class ``GP``).

Same constructor, ``Data_sampling`` / ``GP_initialization`` / ``add_sample`` / ``GP_inference`` and the
same ``inference_datasets`` contract (reference GP_Safe.py:16-23,236-245); arrays are NumPy float64
(jax is not available).  ``GP_inference`` -- the innermost call of every acquisition function -- runs
on the B200 through the C ABI (sbo_point_posterior); there is no CPU inference path.  The
hyper-parameter fit and the normalisation stay on the host, exactly where the reference has them
(GP_Safe.py:84-96,169-234): they are outside the hot path (SURVEY.md section 8d).
"""
from __future__ import annotations

import numpy as np
from scipy.optimize import differential_evolution

from ._boot import package

_EPS_F32 = float(np.finfo(np.float32).eps)
# covariance functions: the reference's 'RBF' (squared exponential) and, additively, Matern 3/2 and 5/2
KERNELS = ('RBF', 'Matern32', 'Matern52')


class GP:
    def __init__(self, plant_system, device=0) -> None:
        self.plant_system = plant_system
        self.n_fun = len(plant_system)
        self.key = np.random.default_rng(42)          # reference: jax.random.PRNGKey(42)
        self.inference_datasets = {"X_mean": [], "X_std": [], "Y_mean": [], "Y_std": [],
                                   "X_norm": [], "Y_norm": [], "invKopt": [], "hypopt": []}
        self.GP_inference_jit = self.GP_inference     # reference: jit(self.GP_inference)
        self.hyper_seed = None                        # set to an int for a reproducible fit
        self.fit_on_device = False                    # additive: evaluate whole DE populations on the GPU (sbo_nll_batch)
        self._device = device
        self._engine = None
        self._uploaded = None                         # id/version of the dataset resident on the GPU
        self._version = 0

    # ------------------------------------------------------------------ engine plumbing
    @property
    def engine(self):
        if self._engine is None:
            self._engine = package().GridEngine(self._device)
        return self._engine

    def _ensure_uploaded(self, ds):
        key = (id(ds), self._version if ds is self.inference_datasets else None,
               id(ds.get("hypopt")), id(ds.get("X_norm")))
        if self._uploaded != key:
            self.engine.set_model(ds, self.kernel)
            self._uploaded = key
            self._on_model_changed()

    def _on_model_changed(self):
        pass

    # ------------------------------------------------------------------ data sampling (GP_Safe.py:29-78)
    def Ball_sampling(self, x_dim, n_sample, r_i, key):
        xi = key.normal(size=(n_sample, x_dim))
        unit = xi / np.linalg.norm(xi, axis=1, keepdims=True)
        u = key.uniform(size=(n_sample, 1))
        return r_i * u ** (1.0 / x_dim) * unit

    def Data_sampling(self, n_sample, x_0, r, noise=0.):
        x_0 = np.asarray(x_0, dtype=np.float64)
        X = self.Ball_sampling(x_0.shape[0], n_sample, r, self.key) + x_0
        Y = np.zeros((n_sample, self.n_fun))
        for i in range(n_sample):
            for j in range(self.n_fun):
                Y[i, j] = self.plant_system[j](X[i], noise)
        return X, Y

    # ------------------------------------------------------------------ host-side GP operations
    def data_normalization(self):
        """GP_Safe.py:84-96."""
        self.X_mean, self.X_std = np.mean(self.X, axis=0), np.std(self.X, axis=0)
        self.Y_mean, self.Y_std = np.mean(self.Y, axis=0), np.std(self.Y, axis=0)
        return (self.X - self.X_mean) / self.X_std, (self.Y - self.Y_mean) / self.Y_std

    def squared_seuclidean_jax(self, X, Y, V):
        """GP_Safe.py:98-120 (name kept for API compatibility)."""
        s = V ** -0.5
        Xa, Ya = X * s, Y * s
        return -2 * np.dot(Xa, Ya.T) + np.sum(Xa ** 2, axis=1)[:, None] + np.sum(Ya ** 2, axis=1)

    def Cov_mat(self, kernel, X_norm, Y_norm, W, sf2):
        """GP_Safe.py:122-143.  s = squared distance scaled by W;  'RBF': sf2 exp(-s/2),  'Matern32': sf2 (1 + t) exp(-t)
        with t = sqrt(3 s),  'Matern52': sf2 (1 + t + t^2/3) exp(-t) with t = sqrt(5 s)."""
        if W.shape[0] != X_norm.shape[1]:
            raise ValueError('ERROR W and X_norm dimension should be same')
        elif kernel not in KERNELS:
            raise ValueError('ERROR no kernel with name ', kernel)
        s = self.squared_seuclidean_jax(X_norm, Y_norm, W)
        if kernel == 'RBF':
            return sf2 * np.exp(-0.5 * s)
        t = np.sqrt((3.0 if kernel == 'Matern32' else 5.0) * np.maximum(s, 0.0))   # the expanded square can round below 0
        poly = 1.0 + t if kernel == 'Matern32' else 1.0 + t + t * t / 3.0
        return sf2 * poly * np.exp(-t)

    def calc_Cov_mat(self, kernel, X_norm, x_norm, ell, sf2):
        """GP_Safe.py:146-167."""
        x_norm = np.asarray(x_norm).reshape(1, self.nx_dim)
        return self.Cov_mat(kernel, X_norm, x_norm, ell, sf2)

    def negative_loglikelihood(self, hyper, X, Y):
        """GP_Safe.py:169-192."""
        d = self.nx_dim
        W, sf2, sn2 = np.exp(2 * hyper[:d]), np.exp(2 * hyper[d]), np.exp(2 * hyper[d + 1])
        K = self.Cov_mat(self.kernel, X, X, W, sf2) + (sn2 + 1e-8) * np.eye(X.shape[0])
        K = (K + K.T) * 0.5
        try:
            L = np.linalg.cholesky(K)
        except np.linalg.LinAlgError:
            return 1e30
        logdetK = 2 * np.sum(np.log(np.diag(L)))
        a = np.linalg.solve(L.T, np.linalg.solve(L, Y))
        return float(np.dot(Y.T, a)[0][0] + logdetK)

    def determine_hyperparameters(self, X_norm, Y_norm):
        """GP_Safe.py:194-234: per-output differential evolution; returns (hypopt, invKopt)."""
        d = self.nx_dim
        bounds = [(-1.5, 1.5)] * (d + 1) + [(-5., -2.)]
        hypopt = np.zeros((d + 2, self.ny_dim))
        invKopt = []
        for i in range(self.ny_dim):
            kw = {} if self.hyper_seed is None else {"seed": self.hyper_seed + i}
            if self.fit_on_device:
                # same objective and bounds, but SciPy hands over the whole population (d+2, S) per generation and the
                # GPU factorises the S covariance matrices in one batch; 'deferred' updating is what vectorised
                # evaluation implies, so the search path (not the objective) differs from the reference's
                yi = np.ascontiguousarray(Y_norm[:, i])
                res = differential_evolution(lambda H: self.engine.nll_batch(X_norm, yi, np.atleast_2d(H.T), self.kernel),
                                             bounds=bounds, vectorized=True, updating='deferred', **kw)
            else:
                res = differential_evolution(self.negative_loglikelihood, args=(X_norm, Y_norm[:, i:i + 1]),
                                             bounds=bounds, **kw)
            hypopt[:, i] = res.x
            ellopt = np.exp(2. * hypopt[:d, i])
            sf2opt = np.exp(2. * hypopt[d, i])
            sn2opt = np.exp(2. * hypopt[d + 1, i]) + _EPS_F32
            Kopt = self.Cov_mat(self.kernel, X_norm, X_norm, ellopt, sf2opt) + sn2opt * np.eye(self.n_point)
            invKopt += [np.linalg.inv(Kopt)]
        return hypopt, invKopt

    def update_inference_dataset(self):
        """GP_Safe.py:236-245."""
        ds = self.inference_datasets
        ds["X_mean"], ds["X_std"] = self.X_mean, self.X_std
        ds["Y_mean"], ds["Y_std"] = self.Y_mean, self.Y_std
        ds["X_norm"], ds["Y_norm"] = self.X_norm, self.Y_norm
        ds["invKopt"], ds["hypopt"] = self.invKopt, self.hypopt
        self._version += 1

    def set_hyperparameters(self, hypopt):
        """Additive helper: install fixed hyper-parameters instead of fitting (fixtures, benchmarks)."""
        self.hypopt = np.asarray(hypopt, dtype=np.float64)
        d = self.nx_dim
        self.invKopt = []
        for i in range(self.ny_dim):
            K = self.Cov_mat(self.kernel, self.X_norm, self.X_norm, np.exp(2. * self.hypopt[:d, i]),
                             np.exp(2. * self.hypopt[d, i]))
            K = K + (np.exp(2. * self.hypopt[d + 1, i]) + _EPS_F32) * np.eye(self.n_point)
            self.invKopt.append(np.linalg.inv(K))
        self.update_inference_dataset()

    # ------------------------------------------------------------------ initialisation / update
    def GP_initialization(self, X, Y, kernel, multi_hyper, var_out=True, hypopt=None):
        """GP_Safe.py:251-277.  ``kernel``: 'RBF' as in the reference, or (additive) 'Matern32' / 'Matern52'.
        ``hypopt`` (additive, optional) skips the fit."""
        self.X, self.Y, self.kernel = np.asarray(X, dtype=np.float64), np.asarray(Y, dtype=np.float64), kernel
        if kernel not in KERNELS:
            raise ValueError('ERROR no kernel with name ', kernel)
        self.n_point, self.nx_dim = self.X.shape[0], self.X.shape[1]
        self.ny_dim = self.Y.shape[1]
        self.multi_hyper = multi_hyper
        self.var_out = var_out
        self.X_norm, self.Y_norm = self.data_normalization()
        if hypopt is not None:
            self.set_hyperparameters(hypopt)
        else:
            self.hypopt, self.invKopt = self.determine_hyperparameters(self.X_norm, self.Y_norm)
            self.update_inference_dataset()

    def add_sample(self, x_new, y_new, hypopt=None):
        """GP_Safe.py:283-304: append, re-normalise, refit everything."""
        self.X = np.vstack([self.X, np.asarray(x_new, dtype=np.float64)])
        self.Y = np.vstack([self.Y, np.asarray(y_new, dtype=np.float64)])
        self.n_point = self.X.shape[0]
        self.X_norm, self.Y_norm = self.data_normalization()
        if hypopt is not None:
            self.set_hyperparameters(hypopt)
        else:
            self.hypopt, self.invKopt = self.determine_hyperparameters(self.X_norm, self.Y_norm)
            self.update_inference_dataset()

    def add_sample_fixed(self, x_new, y_new):
        """Additive (SURVEY.md section 8f row 1): one more observation at FIXED hyper-parameters and FIXED
        normalisation constants -- what a controller does between two re-fits.  The device appends one row to the
        Cholesky factor and refreshes W = L^-1 and alpha in O(n^2) (``sbo_append_sample``); nothing is re-uploaded and
        the O(n^3) ``inv(K)`` of GP_Safe.py:232 is not formed (``invKopt`` is dropped from ``inference_datasets``:
        the grid path never reads it).  ``add_sample`` keeps the reference's re-fit + re-normalise semantics."""
        self._ensure_uploaded(self.inference_datasets)
        x_new = np.asarray(x_new, dtype=np.float64).reshape(1, -1)
        y_new = np.asarray(y_new, dtype=np.float64).reshape(1, -1)
        xn, yn = (x_new - self.X_mean) / self.X_std, (y_new - self.Y_mean) / self.Y_std
        self.engine.append_sample(xn, yn)
        self.X, self.Y = np.vstack([self.X, x_new]), np.vstack([self.Y, y_new])
        self.X_norm, self.Y_norm = np.vstack([self.X_norm, xn]), np.vstack([self.Y_norm, yn])
        self.n_point = self.X.shape[0]
        self.invKopt = None
        self.update_inference_dataset()
        ds = self.inference_datasets                    # the device already holds this state: no upload on the next call
        self._uploaded = (id(ds), self._version, id(ds.get("hypopt")), id(ds.get("X_norm")))
        self._on_model_appended()

    def _on_model_appended(self):
        """The device model gained samples through sbo_append_sample only (subclasses may update instead of recompute)."""
        self._on_model_changed()

    # ------------------------------------------------------------------ inference (GPU)
    def GP_inference(self, x, inference_dataset):
        """GP_Safe.py:310-352 on the B200: returns (mean (G,), var (G,)), or mean[0] if not var_out."""
        self._ensure_uploaded(inference_dataset)
        mean, var = self.engine.point_posterior(np.asarray(x, dtype=np.float64).reshape(1, -1))
        if self.var_out:
            return mean[0], var[0]
        return mean.flatten()[0]

    def GP_inference_batch(self, points, inference_dataset=None):
        """Additive: the vmapped form, (m,d) -> (mean (m,G), var (m,G))."""
        self._ensure_uploaded(self.inference_datasets if inference_dataset is None else inference_dataset)
        return self.engine.point_posterior(points)
