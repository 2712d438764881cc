"""GridEngine -- host-side driver of the CUDA grid pipeline (through the C ABI only).

One engine = one ``sbo_ctx`` = one GPU.  It owns no numerics: every number it
returns was produced by a kernel of libsbo_b200.so.  The reference objects it
feeds are the drop-in classes in ``models/`` (SafeOpt.BO, GoOSE.BO).
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _capi as capi


class SboError(RuntimeError):
    pass


def _f64(a):
    return np.ascontiguousarray(np.asarray(a, dtype=np.float64))


def kernel_id(kernel):
    """enum sbo_kernel of a covariance function name ('RBF', 'Matern32', 'Matern52')."""
    if kernel not in capi.KERNELS:
        raise ValueError(f"unknown kernel {kernel!r}: expected one of {', '.join(capi.KERNELS)}")
    return capi.KERNELS[kernel]


def unpack_bits(words, count):
    """uint32 little-endian bit words -> bool array of length count."""
    b = np.unpackbits(np.ascontiguousarray(words).view(np.uint8), bitorder="little")
    return b[:count].astype(bool)


class GridEngine:
    def __init__(self, device=0, stream=None):
        self._lib = capi.load()
        h = C.c_void_p()
        rc = self._lib.sbo_create(int(device), C.byref(h))
        if rc != 0:
            raise SboError(f"sbo_create failed ({rc}): {self._lib.sbo_last_error(None).decode()}")
        self._h = h
        self.device = int(device)
        self.n = self.d = self.G = 0
        self.N = 0
        self.first = 0
        self.count = 0
        self.grid_kind = None
        self.comm_ready = False
        self.options = {}                   # what set_option was called with
        self.stream = None                  # the raw cudaStream_t the context launches on (None = its own stream)
        if stream is not None:
            self._ck(self._lib.sbo_set_stream(self._h, C.c_void_p(int(stream))))
            self.stream = int(stream)
        import os
        for env, opt in (("SBO_FANTASY_VARIANT", "fantasy_variant"), ("SBO_POSTERIOR_VARIANT", "posterior_variant"),
                         ("SBO_FANTASY_GX", "fantasy_gx"), ("SBO_POSTERIOR_CHUNK_MB", "posterior_chunk_mb"),
                         ("SBO_POSTERIOR_FUSED", "posterior_fused"), ("SBO_FANTASY_REFINE", "fantasy_refine"),
                         ("SBO_FANTASY_REFINE_MB", "fantasy_refine_mb"),
                         ("SBO_POSTERIOR_TABLES", "posterior_tables")):
            if os.environ.get(env):
                self.set_option(opt, int(os.environ[env]))

    # -- plumbing ---------------------------------------------------------------------------
    def _ck(self, rc):
        if rc != 0:
            msg = self._lib.sbo_last_error(self._h).decode()
            if rc == -1:
                raise ValueError(msg)
            raise SboError(f"libsbo_b200 error {rc}: {msg}")

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._lib.sbo_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_option(self, name, value):
        self._ck(self._lib.sbo_set_option(self._h, name.encode(), int(value)))
        self.options[name] = int(value)

    def release(self, what=3):
        """Free device workspaces: 1 = per-point V rows, 2 = gathered pair operands, 3 = both (large grids)."""
        self._ck(self._lib.sbo_release(self._h, int(what)))

    def kernel_launches(self, reset=False):
        return int(self._lib.sbo_kernel_launches(self._h, 1 if reset else 0))

    def mem_peak(self, reset=False):
        """High-water mark (bytes) of the device memory of the context's work buffers."""
        return int(self._lib.sbo_mem_peak(self._h, 1 if reset else 0))

    def refine_stats(self):
        """FP64 refinement of the last pair stage: {"cells": cells of the pass, "fp64_rows": FP64 rows computed} (0/0: none)."""
        cells, rows = C.c_int64(), C.c_int64()
        self._ck(self._lib.sbo_refine_stats(self._h, C.byref(cells), C.byref(rows)))
        return {"cells": int(cells.value), "fp64_rows": int(rows.value)}

    def phase_ms(self):
        out = {}
        v = C.c_double()
        for i, nm in enumerate(capi.PHASES):
            self._ck(self._lib.sbo_phase_ms(self._h, i, C.byref(v)))
            out[nm] = v.value
        return out

    # -- model ------------------------------------------------------------------------------
    def set_model(self, ds, kernel="RBF"):
        """Upload ``inference_datasets`` (models/GP_Safe.py:236-245) with the covariance function ``kernel`` ('RBF',
        'Matern32' or 'Matern52').  invKopt is not needed."""
        kid = kernel_id(kernel)
        Xn, Yn, hyp = _f64(ds["X_norm"]), _f64(ds["Y_norm"]), _f64(ds["hypopt"])
        n, d = Xn.shape
        G = Yn.shape[1]
        if hyp.shape != (d + 2, G):
            raise ValueError("ERROR W and X_norm dimension should be same")   # GP_Safe.py:134-135
        xm, xs, ym, ys = _f64(ds["X_mean"]), _f64(ds["X_std"]), _f64(ds["Y_mean"]), _f64(ds["Y_std"])
        self._ck(self._lib.sbo_set_model_ex(self._h, kid, n, d, G, capi.dptr(Xn), capi.dptr(Yn), capi.dptr(xm), capi.dptr(xs),
                                            capi.dptr(ym), capi.dptr(ys), capi.dptr(hyp)))
        self.n, self.d, self.G = n, d, G

    def append_sample(self, x_norm_new, y_norm_new):
        """Rank-1 append at fixed hyper-parameters / normalisation (sbo_append_sample): n -> n + 1."""
        x, y = _f64(x_norm_new).reshape(-1), _f64(y_norm_new).reshape(-1)
        if x.shape[0] != self.d or y.shape[0] != self.G:
            raise ValueError("x_norm_new must have d entries and y_norm_new G entries")
        self._ck(self._lib.sbo_append_sample(self._h, capi.dptr(x), capi.dptr(y)))
        self.n += 1

    def stable_minmax(self, n_controlled, fun="ucb", beta=2.0, want_scores=False):
        """StableOpt on the grid: (x_c index, min over the robust safe set of max_d fun_0, |robust safe set|[, scores])."""
        kind = {"mean": 0, "ucb": 1, "lcb": 2}[fun]
        idx, val, cnt = C.c_int64(), C.c_double(), C.c_int64()
        sc, sp = None, None
        if want_scores:
            sc = np.empty(int(np.prod(self.grid_shape[:n_controlled])))
            sp = capi.dptr(sc)
        self._ck(self._lib.sbo_stable_minmax(self._h, int(n_controlled), kind, float(beta), C.byref(idx), C.byref(val), C.byref(cnt), sp))
        return (idx.value, val.value, cnt.value, sc) if want_scores else (idx.value, val.value, cnt.value)

    def nll_batch(self, X_norm, y, hyp_pop, kernel="RBF"):
        """GP.negative_loglikelihood (GP_Safe.py:169-192) for a population: hyp_pop (P, d+2) -> nll (P,)."""
        kid = kernel_id(kernel)
        Xn, yv, hp = _f64(X_norm), _f64(y).reshape(-1), _f64(hyp_pop)
        n, d = Xn.shape
        if hp.ndim != 2 or hp.shape[1] != d + 2 or yv.shape[0] != n:
            raise ValueError("hyp_pop must be (P, d+2) and y (n,)")
        out = np.empty(hp.shape[0])
        self._ck(self._lib.sbo_nll_batch_ex(self._h, kid, n, d, capi.dptr(Xn), capi.dptr(yv), hp.shape[0], capi.dptr(hp), capi.dptr(out)))
        return out

    def get_model(self):
        L = np.empty((self.G, self.n, self.n))
        W = np.empty((self.G, self.n, self.n))
        a = np.empty((self.G, self.n))
        self._ck(self._lib.sbo_get_model(self._h, capi.dptr(L), capi.dptr(W), capi.dptr(a)))
        return L, W, a

    # -- points -----------------------------------------------------------------------------
    def set_grid(self, lo, hi, pts):
        lo, hi = _f64(lo), _f64(hi)
        pts = np.ascontiguousarray(np.asarray(pts, dtype=np.int64))
        d = lo.shape[0]
        self._ck(self._lib.sbo_set_grid(self._h, d, pts.ctypes.data_as(C.POINTER(C.c_int64)), capi.dptr(lo), capi.dptr(hi)))
        self.N = int(np.prod(pts))
        self.first, self.count = 0, self.N
        self.grid_kind = "mesh"
        self.gd = d
        self.grid_shape = tuple(int(p) for p in pts)

    def set_points(self, pts):
        pts = _f64(pts)
        N, d = pts.shape
        self._ck(self._lib.sbo_set_points(self._h, N, d, capi.dptr(pts)))
        self.N = N
        self.first, self.count = 0, N
        self.grid_kind = "points"
        self.gd = d

    def set_shard(self, first, count):
        self._ck(self._lib.sbo_set_shard(self._h, int(first), int(count)))
        self.first, self.count = int(first), int(count)

    def set_shard_cyclic(self, rank, nranks, block=256):
        """Block-cyclic ownership of the grid (multi-GPU): returns the number of local points."""
        c = C.c_int64()
        self._ck(self._lib.sbo_set_shard_cyclic(self._h, int(rank), int(nranks), int(block), C.byref(c)))
        self.first, self.count = 0, int(c.value)
        return self.count

    def point_coords(self, idx):
        x = np.empty(8)
        self._ck(self._lib.sbo_point_coords(self._h, int(idx), capi.dptr(x)))
        return x[: self.gd].copy()

    # -- posterior --------------------------------------------------------------------------
    def posterior(self, with_grad=False, keep_v=0, fetch=True):
        """GP posterior over the local shard.  Returns (mean, var) as (count, G) views when fetch."""
        if fetch:
            mean = np.empty((self.G, self.count))
            var = np.empty((self.G, self.count))
            self._ck(self._lib.sbo_posterior(self._h, int(with_grad), int(keep_v), capi.dptr(mean), capi.dptr(var)))
            return mean.T, var.T
        self._ck(self._lib.sbo_posterior(self._h, int(with_grad), int(keep_v), None, None))
        return None

    def posterior_update(self, fetch=True):
        """Bring the last posterior up to the model after the append_sample calls made since (sbo_posterior_update), with
        the same with_grad and keep_v.  Returns ((mean, var) as in posterior() or None, info) with info = {"rows": samples
        appended since that posterior, "recomputed": True when the update ran the full posterior (V rows kept and the
        padded factor grew)}.  Raises ValueError when anything else changed the model, grid or shard since."""
        info = capi.UpdateInfo()
        if fetch:
            mean = np.empty((self.G, self.count))
            var = np.empty((self.G, self.count))
            self._ck(self._lib.sbo_posterior_update(self._h, capi.dptr(mean), capi.dptr(var), C.byref(info)))
            out = (mean.T, var.T)
        else:
            self._ck(self._lib.sbo_posterior_update(self._h, None, None, C.byref(info)))
            out = None
        return out, {"rows": int(info.rows), "recomputed": bool(info.recomputed)}

    def point_posterior(self, x):
        x = _f64(x).reshape(-1, self.d)
        m = x.shape[0]
        mean = np.empty((m, self.G))
        var = np.empty((m, self.G))
        self._ck(self._lib.sbo_point_posterior(self._h, m, capi.dptr(x), capi.dptr(mean), capi.dptr(var)))
        return mean, var

    def point_mean_grad(self, x, gp):
        x = _f64(x).reshape(-1, self.d)
        g = np.empty((x.shape[0], self.d))
        self._ck(self._lib.sbo_point_mean_grad(self._h, int(gp), x.shape[0], capi.dptr(x), capi.dptr(g)))
        return g

    def lipschitz(self):
        L = np.empty(self.G)
        self._ck(self._lib.sbo_lipschitz(self._h, capi.dptr(L)))
        return L

    # -- sets -------------------------------------------------------------------------------
    @staticmethod
    def _sets_dict(r):
        return {k: getattr(r, k) for k, _ in capi.SetsResult._fields_}

    def sets(self, beta, unsafe_rule=capi.UNSAFE_ALL, strict=False):
        r = capi.SetsResult()
        self._ck(self._lib.sbo_sets(self._h, float(beta), int(unsafe_rule), int(bool(strict)), C.byref(r)))
        return self._sets_dict(r)

    def sets_pass1(self, beta, unsafe_rule=capi.UNSAFE_ALL, strict=False):
        r = capi.SetsResult()
        self._ck(self._lib.sbo_sets_pass1(self._h, float(beta), int(unsafe_rule), int(bool(strict)), C.byref(r)))
        return self._sets_dict(r)

    def sets_pass2(self, min_ucb0):
        r = capi.SetsResult()
        self._ck(self._lib.sbo_sets_pass2(self._h, float(min_ucb0), C.byref(r)))
        return self._sets_dict(r)

    def mask(self, kind, which=0):
        nw = (self.count + 31) // 32
        w = np.empty(nw, dtype=np.uint32)
        self._ck(self._lib.sbo_get_mask(self._h, int(kind), int(which), w.ctypes.data_as(C.POINTER(C.c_uint32))))
        return unpack_bits(w, self.count)

    def set_user_mask(self, mask_bool):
        m = np.zeros(((self.count + 31) // 32) * 32, dtype=np.uint8)
        m[: self.count] = np.asarray(mask_bool, dtype=np.uint8)
        w = np.packbits(m, bitorder="little").view(np.uint32)
        w = np.ascontiguousarray(w)
        self._ck(self._lib.sbo_set_user_mask(self._h, w.ctypes.data_as(C.POINTER(C.c_uint32))))

    def user_mask_ball(self, x0, r, mask_kind=capi.MASK_SAFE):
        """user mask = mask_kind AND ||x - x0|| <= r, built on the device (sbo_user_mask_ball)."""
        c = _f64(x0).reshape(-1)
        self._ck(self._lib.sbo_user_mask_ball(self._h, int(mask_kind), capi.dptr(c), float(r)))

    def mask_dev(self, kind, which=0):
        p = C.c_void_p()
        n = C.c_int64()
        self._ck(self._lib.sbo_mask_dev(self._h, int(kind), int(which), C.byref(p), C.byref(n)))
        return p.value, n.value

    def posterior_dev(self):
        m, v = C.c_void_p(), C.c_void_p()
        self._ck(self._lib.sbo_posterior_dev(self._h, C.byref(m), C.byref(v)))
        return m.value, v.value

    def argreduce(self, kind, mask_kind, which=0, target=None):
        idx = C.c_int64()
        val = C.c_double()
        t = None
        if target is not None:
            tt = _f64(target)
            t = capi.dptr(tt)
        self._ck(self._lib.sbo_argreduce(self._h, int(kind), int(mask_kind), int(which), t, C.byref(idx), C.byref(val)))
        return idx.value, val.value

    # -- pair kernels -----------------------------------------------------------------------
    def _pair_dict(self, r):
        nc = max(self.G - 1, 0)
        return {"best_idx": r.best_idx, "best_value": r.best_value,
                "per_idx": [r.per_idx[c] for c in range(nc)], "per_value": [r.per_value[c] for c in range(nc)],
                "n_x": r.n_x, "n_z": r.n_z, "pairs_algorithmic": r.pairs_algorithmic,
                "pairs_evaluated": r.pairs_evaluated, "n_hit": r.n_hit, "n_ambiguous": r.n_ambiguous,
                "n_refined_safe": r.n_refined_safe, "n_undecided": r.n_undecided,
                "undecided_best_idx": r.undecided_best_idx, "undecided_best_value": r.undecided_best_value}

    def expander(self, beta, L=None, mode=capi.MODE_LIPSCHITZ, precision=capi.PREC_FP64, want_counts=False):
        r = capi.PairResult()
        Lp = None
        if L is not None:
            Lc = _f64(L)
            if Lc.shape[0] != self.G:
                raise ValueError("L must have one entry per GP")
            Lp = capi.dptr(Lc)
        counts = None
        cp = None
        if want_counts and mode == capi.MODE_FANTASY:
            counts = np.zeros(self.count, dtype=np.int32)
            cp = counts.ctypes.data_as(C.POINTER(C.c_int32))
        self._ck(self._lib.sbo_expander(self._h, int(mode), int(precision), float(beta), Lp, C.byref(r), cp))
        out = self._pair_dict(r)
        if counts is not None:
            out["counts"] = counts
        return out

    def goose_target(self, beta, L=None, mode=capi.MODE_LIPSCHITZ, precision=capi.PREC_FP64):
        """GoOSE target set (SBO_MASK_TARGET) and its argmin lcb_0: Lipschitz pair test (L required) or fantasy test."""
        r = capi.PairResult()
        Lp = None
        if mode == capi.MODE_LIPSCHITZ or L is not None:
            Lc = _f64(L)
            if Lc.ndim != 1 or Lc.shape[0] != self.G:
                raise ValueError("L must have one entry per GP")
            Lp = capi.dptr(Lc)
        self._ck(self._lib.sbo_goose_target_ex(self._h, int(mode), int(precision), float(beta), Lp, C.byref(r)))
        return self._pair_dict(r)

    # -- staged pair driver (multi-GPU; tensors are torch CUDA tensors or anything with data_ptr()) --------
    @staticmethod
    def _ptr(t):
        if t is None:
            return None
        return C.c_void_p(int(t.data_ptr())) if hasattr(t, "data_ptr") else C.c_void_p(int(t))

    def pairs_prepare(self, mode, precision, beta, L=None):
        info = capi.PairsInfo()
        Lp = None
        if L is not None:
            Lc = _f64(L)
            Lp = capi.dptr(Lc)
        self._ck(self._lib.sbo_pairs_prepare(self._h, int(mode), int(precision), float(beta), Lp, C.byref(info)))
        return {k: getattr(info, k) for k, _ in capi.PairsInfo._fields_}

    def pairs_export(self, rows, vrows=None):
        self._ck(self._lib.sbo_pairs_export_dev(self._h, self._ptr(rows), self._ptr(vrows)))

    def pairs_import(self, n_total, rows, vrows=None):
        self._ck(self._lib.sbo_pairs_import_dev(self._h, int(n_total), self._ptr(rows), self._ptr(vrows)))

    def pairs_set_segments(self, n_per_rank, rank):
        n = np.ascontiguousarray(np.asarray(n_per_rank, dtype=np.int64))
        self._ck(self._lib.sbo_pairs_set_segments(self._h, int(n.size), int(rank), n.ctypes.data_as(C.POINTER(C.c_int64))))

    def mask_export(self, kind, dst, which=0):
        """Copy a local bitmask into a caller-owned device buffer of int32/uint32 words (zero padded)."""
        self._ck(self._lib.sbo_mask_export_dev(self._h, int(kind), int(which), self._ptr(dst), int(dst.numel())))

    def pairs_set_global_unsafe(self, gathered, words_per_rank, nranks):
        self._ck(self._lib.sbo_pairs_set_global_unsafe_dev(self._h, self._ptr(gathered), int(words_per_rank), int(nranks)))

    def pairs_run(self, goose, result):
        self._ck(self._lib.sbo_pairs_run_dev(self._h, int(bool(goose)), self._ptr(result)))

    def pairs_finish(self, goose, offset, result, want_counts=False):
        r = capi.PairResult()
        counts, cp = None, None
        if want_counts:
            counts = np.zeros(self.count, dtype=np.int32)
            cp = counts.ctypes.data_as(C.POINTER(C.c_int32))
        self._ck(self._lib.sbo_pairs_finish_dev(self._h, int(bool(goose)), int(offset), self._ptr(result), C.byref(r), cp))
        out = self._pair_dict(r)
        if counts is not None:
            out["counts"] = counts
        return out

    # -- library-owned communicator + whole sharded steps (csrc/comm.cu) ---------------------------------
    def comm_unique_id(self):
        buf = (C.c_char * 128)()
        self._ck(self._lib.sbo_comm_unique_id(C.cast(buf, C.c_void_p)))
        return bytes(buf)

    def comm_init(self, rank, nranks, unique_id):
        buf = (C.c_char * 128).from_buffer_copy(bytes(unique_id))
        self._ck(self._lib.sbo_comm_init(self._h, int(rank), int(nranks), C.cast(buf, C.c_void_p)))
        self.comm_ready = True

    def _step_dict(self, r, goose):
        out = self._sets_dict(r.sets)
        out["L"] = np.array([r.L[i] for i in range(self.G)])
        pr = self._pair_dict(r.pairs)
        out["x_new_idx"], out["explore_idx"] = r.x_new_idx, r.explore_idx
        if goose:
            out["target"] = pr
            out["target_idx"], out["target_lcb"] = pr["best_idx"], pr["best_value"]
        else:
            out["expander"] = pr
            out["expander_idx"] = pr["best_idx"]
            out["expander_std"] = float(np.sqrt(pr["best_value"])) if pr["best_idx"] >= 0 else 0.0
            out["minimizer_std"] = float(np.sqrt(out["minimizer_var"])) if out["minimizer_idx"] >= 0 else 0.0
        return out

    def safeopt_step_sharded(self, ds, beta, mode="lipschitz", precision="fp64", unsafe_rule=capi.UNSAFE_ALL, L=None, upload=True,
                             kernel="RBF"):
        """One SafeOpt step on a grid sharded over the ranks of the library's communicator (sbo_comm_init); the
        collectives run inside the library.  Every rank returns the same global result."""
        if upload:
            self.set_model(ds, kernel)
        prec, _ = capi.PRECISIONS[precision]
        r = capi.StepResult()
        Lp = capi.dptr(_f64(L)) if L is not None else None
        self._ck(self._lib.sbo_safeopt_step_sharded(self._h, float(beta), capi.MODE_FANTASY if mode == "fantasy" else capi.MODE_LIPSCHITZ,
                                                    int(prec), int(unsafe_rule), Lp, C.byref(r)))
        return self._step_dict(r, False)

    def goose_step_sharded(self, ds, beta, unsafe_rule=capi.UNSAFE_ALL, L=None, upload=True, mode="lipschitz", precision="fp64",
                           kernel="RBF"):
        if upload:
            self.set_model(ds, kernel)
        prec, _ = capi.PRECISIONS[precision]
        r = capi.StepResult()
        Lp = capi.dptr(_f64(L)) if L is not None else None
        self._ck(self._lib.sbo_goose_step_sharded_ex(self._h, float(beta), capi.MODE_FANTASY if mode == "fantasy" else capi.MODE_LIPSCHITZ,
                                                     int(prec), int(unsafe_rule), Lp, C.byref(r)))
        return self._step_dict(r, True)

    # -- batch SafeOpt acquisition (csrc/batch.cu): q safe query points per step ----------------------------------------
    @staticmethod
    def _pick_dict(p):
        return {k: getattr(p, k) for k, _ in capi.BatchPick._fields_ if k != "pad"}

    def safeopt_batch(self, q):
        """q query points from the last SafeOpt step (sbo_safeopt_batch): a list of n_picked dicts with idx (global),
        from_expander, std_min / idx_min and std_exp / idx_exp under the earlier picks; empty when M and E are empty."""
        q = int(q)
        arr = (capi.BatchPick * max(q, 1))()
        n = C.c_int()
        self._ck(self._lib.sbo_safeopt_batch(self._h, q, arr, C.byref(n)))
        return [self._pick_dict(arr[b]) for b in range(n.value)]

    def safeopt_batch_sharded(self, q):
        """safeopt_batch on a grid sharded over the library's communicator (sbo_comm_init); every rank gets the same picks."""
        q = int(q)
        arr = (capi.BatchPick * max(q, 1))()
        n = C.c_int()
        self._ck(self._lib.sbo_safeopt_batch_sharded(self._h, q, arr, C.byref(n)))
        return [self._pick_dict(arr[b]) for b in range(n.value)]

    def batch_prepare(self, q):
        """Staged batch, step 1: compact this shard's candidates M u E; returns their number."""
        n = C.c_int64()
        self._ck(self._lib.sbo_batch_prepare(self._h, int(q), C.byref(n)))
        return int(n.value)

    def batch_local(self):
        """Staged batch, step 2: this shard's optima for the next pick (global indices)."""
        p = capi.BatchPick()
        self._ck(self._lib.sbo_batch_local(self._h, C.byref(p)))
        return self._pick_dict(p)

    def batch_commit(self, global_idx):
        """Staged batch, step 3: hallucinate an observation at the chosen global index."""
        self._ck(self._lib.sbo_batch_commit(self._h, int(global_idx)))

    # -- batch GoOSE acquisition (csrc/batch.cu): q distinct safe query points per step ---------------------------------
    @staticmethod
    def _goose_pick_dict(p):
        return {k: getattr(p, k) for k, _ in capi.GooseBatchPick._fields_ if k != "pad"}

    def goose_batch(self, q):
        """q query points from the last GoOSE step (sbo_goose_batch): a list of min(q, |S|) dicts with idx (global), explore,
        safe_lcb / safe_idx and target_lcb / target_idx under the earlier picks, and dist (explore picks)."""
        q = int(q)
        arr = (capi.GooseBatchPick * max(q, 1))()
        n = C.c_int()
        self._ck(self._lib.sbo_goose_batch(self._h, q, arr, C.byref(n)))
        return [self._goose_pick_dict(arr[b]) for b in range(n.value)]

    def goose_batch_sharded(self, q):
        """goose_batch on a grid sharded over the library's communicator (sbo_comm_init); every rank gets the same picks."""
        q = int(q)
        arr = (capi.GooseBatchPick * max(q, 1))()
        n = C.c_int()
        self._ck(self._lib.sbo_goose_batch_sharded(self._h, q, arr, C.byref(n)))
        return [self._goose_pick_dict(arr[b]) for b in range(n.value)]

    def goose_batch_prepare(self, q):
        """Staged GoOSE batch, step 1: compact this shard's candidates S u T; returns their number."""
        n = C.c_int64()
        self._ck(self._lib.sbo_goose_batch_prepare(self._h, int(q), C.byref(n)))
        return int(n.value)

    def goose_batch_local(self):
        """Staged GoOSE batch, step 2: this shard's (safe, target) optima for the next pick (global indices); idx is -1 for an
        explore pick, whose point goose_batch_nearest finds."""
        p = capi.GooseBatchPick()
        self._ck(self._lib.sbo_goose_batch_local(self._h, C.byref(p)))
        return self._goose_pick_dict(p)

    def goose_batch_nearest(self, target_idx):
        """Staged GoOSE batch, explore picks: this shard's remaining safe point nearest to the global target index ->
        (global index, squared distance); (-1, inf) when none is left here."""
        i, d2 = C.c_int64(), C.c_double()
        self._ck(self._lib.sbo_goose_batch_nearest(self._h, int(target_idx), C.byref(i), C.byref(d2)))
        return int(i.value), float(d2.value)

    def goose_batch_commit(self, pick_idx, served_target_idx=-1):
        """Staged GoOSE batch, step 3: hallucinate an observation at the pick and retire it and the target it served
        (-1: a safe pick)."""
        self._ck(self._lib.sbo_goose_batch_commit(self._h, int(pick_idx), int(served_target_idx)))

    # -- whole steps (drivers' decision rules) ------------------------------------------------
    def safeopt_step(self, ds, beta, mode="lipschitz", precision="fp64", unsafe_rule=capi.UNSAFE_ALL, L=None,
                     upload=True, kernel="RBF"):
        """model upload -> posterior -> sets -> L -> expander pairs -> arg-reductions -> x_new.
        Decision rule of test/test_SafeOpt.py:144-158.  Returns a dict of scalars/indices."""
        if upload:
            self.set_model(ds, kernel)
        fantasy = mode == "fantasy"
        prec, kv = capi.PRECISIONS[precision]
        keep_v = kv if fantasy else 0
        self.posterior(with_grad=not fantasy and L is None, keep_v=keep_v, fetch=False)
        s = self.sets(beta, unsafe_rule)
        out = dict(s)
        out["minimizer_std"] = float(np.sqrt(s["minimizer_var"])) if s["minimizer_idx"] >= 0 else 0.0
        if fantasy:
            ex = self.expander(beta, None, capi.MODE_FANTASY, prec)
        else:
            if L is None:
                Lg = self.lipschitz()
                L = np.full(self.G, Lg[self.G - 1])       # SafeOpt.py:110: L of constraint n_fun-1 for every idx
                out["L"] = Lg
            ex = self.expander(beta, L, capi.MODE_LIPSCHITZ, prec)
        out["expander"] = ex
        out["expander_idx"] = ex["best_idx"]
        out["expander_std"] = float(np.sqrt(ex["best_value"])) if ex["best_idx"] >= 0 else 0.0
        out["x_new_idx"] = s["minimizer_idx"] if out["minimizer_std"] > out["expander_std"] else ex["best_idx"]
        return out

    def goose_step(self, ds, beta, unsafe_rule=capi.UNSAFE_ALL, L=None, upload=True, mode="lipschitz", precision="fp64",
                   kernel="RBF"):
        """Decision rule of test/test_GoOSE.py:151-162.  mode="fantasy": the target set comes from the fantasy pair test
        (GP update with y_i = ucb_i(x)) at `precision`; L is not used."""
        if upload:
            self.set_model(ds, kernel)
        fantasy = mode == "fantasy"
        prec, kv = capi.PRECISIONS[precision]
        self.posterior(with_grad=not fantasy and L is None, keep_v=kv if fantasy else 0, fetch=False)
        s = self.sets_pass1(beta, unsafe_rule)
        out = dict(s)
        if fantasy:
            tg = self.goose_target(beta, None, capi.MODE_FANTASY, prec)
        else:
            if L is None:
                Lg = self.lipschitz()
                L = np.full(self.G, Lg[self.G - 1])       # GoOSE.py:100
                out["L"] = Lg
            tg = self.goose_target(beta, L)
        out["target"] = tg
        out["target_idx"], out["target_lcb"] = tg["best_idx"], tg["best_value"]
        if s["min_lcb0"] <= tg["best_value"] or tg["best_idx"] < 0:
            out["x_new_idx"] = s["min_lcb0_idx"]
            out["explore_idx"] = -1
        else:
            e_idx, _ = self.argreduce(capi.ARGMIN_DIST, capi.MASK_SAFE, 0, self.point_coords(tg["best_idx"]))
            out["x_new_idx"] = e_idx
            out["explore_idx"] = e_idx
        return out
