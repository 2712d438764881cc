"""FP64 references for tests/test_gpu_large_n.py at training sets of thousands of samples.

NumPy side: the covariance matrix is built one input dimension at a time (an n x n array at a time, not the (n, n, d) array
of oracle.sq_dist_direct), so n = 8192 needs a few hundred MB of host memory per matrix.  Torch side: the same arithmetic in
float64 on a CUDA device through cuBLAS / cuSOLVER, which share no code with this library; used where the NumPy reference
would take minutes on the host (n = 16384).  Covariance functions as tests/matern_ref.py; the torch side covers SE only."""
from __future__ import annotations

import numpy as np
import scipy.linalg as sla

import matern_ref as R
from oracle import gp_oracle as O

U = 2.0 ** -53          # unit roundoff of FP64


def sq_dist(A, B, ell):
    s = np.zeros((A.shape[0], B.shape[0]))
    for k in range(A.shape[1]):
        df = A[:, k][:, None] - B[:, k][None, :]
        s += df * df / ell[k]
    return s


def build_K(X, ell, sf2, noise, kernel):
    """k(X, X) + noise I in FP64 on the host."""
    K = R.kval(sq_dist(X, X, ell), sf2, kernel)
    K[np.diag_indices_from(K)] += noise
    return K


def model_K(ds, i, kernel):
    d = ds["X_norm"].shape[1]
    ell, sf2, sn2 = O.unpack_hyper(ds["hypopt"][:, i], d)
    return build_K(ds["X_norm"], ell, sf2, sn2 + O.EPS_F32, kernel)


def kappa_bound(ds, i):
    """Upper bound of the 2-norm condition number of K_i: k(X, X) is positive semi-definite, so lambda_min >= sn2 + eps_f32,
    and lambda_max <= n sf2 + sn2 + eps_f32 (Gershgorin)."""
    n, d = ds["X_norm"].shape
    _, sf2, sn2 = O.unpack_hyper(ds["hypopt"][:, i], d)
    noise = sn2 + O.EPS_F32
    return (n * sf2 + noise) / noise


def nll(hyper, X, y, kernel):
    """oracle.negative_loglikelihood (GP_Safe.py:169-192) for any covariance function, with the K built here."""
    d = X.shape[1]
    K = build_K(X, np.exp(2.0 * hyper[:d]), np.exp(2.0 * hyper[d]), np.exp(2.0 * hyper[d + 1]) + 1e-8, kernel)
    L = np.linalg.cholesky(K)
    t = sla.solve_triangular(L, y, lower=True)
    return float(t @ t + 2.0 * np.sum(np.log(np.diag(L))))


def fantasy_margins(xs_pts, zs_pts, ds, beta, kernel, factors, block=4096):
    """Per (z, x) pair min over constraints of (mu' - beta sigma') in normalised units, (|zs|, |xs|), with the V rows of the
    unsafe points computed block by block (R.fantasy_counts_at's arithmetic; counts = (margins >= 0).sum(axis=0))."""
    G, d = ds["Y_norm"].shape[1], xs_pts.shape[1]
    mx, vx, Vx = R.posterior_chol(xs_pts, ds, kernel, return_V=True, factors=factors)
    xn = (xs_pts - ds["X_mean"]) / ds["X_std"]
    out = np.full((zs_pts.shape[0], xs_pts.shape[0]), np.inf)
    for s in range(0, zs_pts.shape[0], block):
        zb = zs_pts[s:s + block]
        mz, vz, Vz = R.posterior_chol(zb, ds, kernel, return_V=True, factors=factors)
        zn = (zb - ds["X_mean"]) / ds["X_std"]
        for i in range(1, G):
            ell, sf2, sn2 = O.unpack_hyper(ds["hypopt"][:, i], d)
            ys2 = ds["Y_std"][i] ** 2
            c = R.kval(sq_dist(zn, xn, ell), sf2, kernel) - Vz[i] @ Vx[i].T
            den = vx[:, i] / ys2 + sn2 + O.EPS_F32
            mu_p = (mz[:, i] / ds["Y_std"][i])[:, None] + c * (beta * np.sqrt(vx[:, i] / ys2) / den)[None, :]
            s2_p = (vz[:, i] / ys2)[:, None] - c * c / den[None, :]
            out[s:s + block] = np.minimum(out[s:s + block], mu_p - beta * np.sqrt(np.maximum(s2_p, 0.0)))
    return out


class TorchSE:
    """FP64 SE-model reference on a CUDA device: K_i, its Cholesky factor and alpha per GP (cuSOLVER), posterior, V rows and
    mean gradients at given points.  Holds G n x n float64 factors on the device."""

    def __init__(self, ds, device="cuda"):
        import torch
        self.t, self.dev = torch, device
        self.ds = ds
        self.n, self.d = ds["X_norm"].shape
        self.G = ds["Y_norm"].shape[1]
        self.X = torch.from_numpy(np.ascontiguousarray(ds["X_norm"])).to(device)
        m0 = O.prior_mean(ds)
        self.hyp = [O.unpack_hyper(ds["hypopt"][:, i], self.d) for i in range(self.G)]
        self.L, self.alpha = [], []
        for i in range(self.G):
            L = torch.linalg.cholesky(self.K(i))
            r = torch.from_numpy(ds["Y_norm"][:, i] - m0[i]).to(device)[:, None]
            self.alpha.append(torch.cholesky_solve(r, L)[:, 0])
            self.L.append(L)
        self.m0 = m0

    def cross(self, A, B, i):
        ell, sf2, _ = self.hyp[i]
        s = self.t.zeros((A.shape[0], B.shape[0]), dtype=self.t.float64, device=self.dev)
        for k in range(self.d):
            df = A[:, k][:, None] - B[:, k][None, :]
            s += df * df / float(ell[k])
        return sf2 * self.t.exp(-0.5 * s)

    def K(self, i):
        _, _, sn2 = self.hyp[i]
        K = self.cross(self.X, self.X, i)
        K.diagonal().add_(sn2 + O.EPS_F32)
        return K

    def _xn(self, pts):
        return self.t.from_numpy((np.atleast_2d(pts) - self.ds["X_mean"]) / self.ds["X_std"]).to(self.dev)

    def posterior(self, pts, i, return_V=False):
        """(mean, var[, V rows (|pts|, n)]) of GP i in raw units, NumPy arrays."""
        ds = self.ds
        _, sf2, _ = self.hyp[i]
        k = self.cross(self.X, self._xn(pts), i)
        v = self.t.linalg.solve_triangular(self.L[i], k, upper=False)
        mean = (self.m0[i] + k.T @ self.alpha[i]) * ds["Y_std"][i] + ds["Y_mean"][i]
        var = self.t.clamp(sf2 - (v * v).sum(0), min=0.0) * ds["Y_std"][i] ** 2
        out = (mean.cpu().numpy(), var.cpu().numpy())
        return out + (v.T.cpu().numpy(),) if return_V else out

    def mean_grad(self, pts, i, block=2048):
        """d mu_i / d x in raw units (R.mean_grad's formula), (|pts|, d)."""
        ds = self.ds
        ell, _, _ = self.hyp[i]
        out = np.empty((np.atleast_2d(pts).shape[0], self.d))
        for s in range(0, out.shape[0], block):
            xn = self._xn(pts[s:s + block])
            w = self.cross(self.X, xn, i) * self.alpha[i][:, None]
            for kk in range(self.d):
                diff = xn[:, kk][None, :] - self.X[:, kk][:, None]
                g = -(w * diff).sum(0) / float(ell[kk]) * ds["Y_std"][i] / ds["X_std"][kk]
                out[s:s + block, kk] = g.cpu().numpy()
        return out
