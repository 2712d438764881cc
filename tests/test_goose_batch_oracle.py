"""CPU: the batch GoOSE acquisition's math and host logic -- the incremental lcb_0 against brute-force augmentation for every
covariance function, pick 1 against the oracle's GoOSE step, distinct picks, short and empty batches, the pick rule on
hand-made sets, the batch driver loop with a stub BO, and the C layout of sbo_goose_batch_pick against its ctypes mirror."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import goose_batch_ref as GB
import matern_ref as MR
import safeopt_batch_ref as SB
from conftest import ROOT, golden_ds, load_golden

Q = 12
SMALL = [(3, 14, 70, 3, "all", 33), (4, 9, 200, 4, "any", 34), (6, 5, 130, 3, "any", 26)]   # as test_gpu_goose_batch.py
GOLD = [("c1_benoit", 9, 3.0, [48, 40], "all"), ("c3_wor", 20, 2.0, [45, 61], "any")]


def _case(name):
    from oracle import gp_oracle as O
    from sbo_b200 import workloads
    if name.startswith("small"):
        d, ppd, n, G, rule, seed = SMALL[int(name[-1])]
        ds, lo, hi, pts, beta = workloads.small(d=d, pts_per_dim=ppd, n=n, seed=seed, G=G)
        # the oracle's own data set (its Lipschitz constants need the inverse Gram matrices)
        ds = O.make_inference_datasets(ds["X_norm"] * ds["X_std"] + ds["X_mean"], ds["Y_norm"] * ds["Y_std"] + ds["Y_mean"], ds["hypopt"])
        return ds, O.make_grid(lo, hi, pts), beta, rule
    gname, n, beta, grid, rule = next(g for g in GOLD if g[0] == name)
    gold = load_golden(gname)
    return golden_ds(O, gold, n), O.make_grid(gold["lo"], gold["hi"], grid), beta, rule


def _oracle_step(name):
    from oracle import gp_oracle as O
    ds, P, beta, rule = _case(name)
    st = O.goose_step(P, ds, beta, unsafe_rule=rule, form="chol")
    T = np.zeros(P.shape[0], dtype=bool)
    for m in st["target_masks"]:
        T |= m
    return ds, P, beta, st, T


@pytest.mark.parametrize("kernel", MR.KERNELS)
def test_incremental_lcb_equals_bruteforce_augmentation(kernel):
    from oracle import gp_oracle as O
    ds, P, beta, _ = _case("small0")
    mean, var = MR.posterior_chol(P, ds, kernel)
    lcb = mean[:, 0] - beta * np.sqrt(var[:, 0])
    S = lcb >= np.quantile(lcb, 0.6)                    # hand-made S and T: what matters is C = S u T
    T = np.zeros_like(S)
    T[np.flatnonzero(~S)[::5]] = True
    hist = []
    picks = GB.goose_batch(P, ds, mean[:, 0], var[:, 0], beta, S, T, 6, kernel=kernel, history=hist)
    assert len(picks) == 6 and any(p["explore"] for p in picks)
    scale = float(np.max(np.abs(lcb[S | T])))
    for b, (cand, got) in enumerate(hist):
        v = SB.variance_bruteforce(P[cand], ds, P[[p["idx"] for p in picks[:b]]], kernel) if b else var[cand, 0]
        ref = mean[cand, 0] - beta * np.sqrt(v)
        assert np.max(np.abs(got - ref)) <= 1e-12 * scale, (kernel, b)
    assert O.masked_argmin(lcb, S)[0] == picks[0]["safe_idx"]


@pytest.mark.parametrize("name", ["small0", "small1", "c1_benoit", "c3_wor"])
def test_pick_one_is_the_oracle_step_and_picks_are_distinct(name):
    ds, P, beta, st, T = _oracle_step(name)
    picks = GB.goose_batch(P, ds, st["mean"][:, 0], st["var"][:, 0], beta, st["S"], T, Q)
    assert len(picks) == min(Q, int(st["S"].sum()))
    p = picks[0]
    assert p["idx"] == st["x_new_idx"]
    assert (p["idx"] if p["explore"] else -1) == st["explore_idx"]
    assert p["safe_lcb"] == st["safe_min_lcb"] and p["target_lcb"] == st["target_lcb"]
    assert len({p["idx"] for p in picks}) == len(picks)
    assert all(st["S"][p["idx"]] for p in picks)
    served = [p["target_idx"] for p in picks if p["explore"]]
    assert len(set(served)) == len(served)
    print(name, "".join("E" if p["explore"] else "S" for p in picks), [p["idx"] for p in picks])


def test_short_and_empty_batches():
    ds, P, beta, st, T = _oracle_step("small2")
    assert st["S"].sum() == 0
    assert GB.goose_batch(P, ds, st["mean"][:, 0], st["var"][:, 0], beta, st["S"], T, 4) == []
    ds, P, beta, st, T = _oracle_step("small0")
    S = np.zeros_like(st["S"])
    S[np.flatnonzero(st["S"])[:3]] = True               # |S| = 3 < q
    picks = GB.goose_batch(P, ds, st["mean"][:, 0], st["var"][:, 0], beta, S, T, 8)
    assert sorted(p["idx"] for p in picks) == list(np.flatnonzero(S))


def test_pick_rule_empty_target_and_equal_lcbs():
    P = np.arange(6, dtype=np.float64)[:, None]
    S = np.array([1, 1, 1, 0, 0, 0], dtype=bool)
    T = np.array([0, 0, 0, 1, 1, 0], dtype=bool)
    none = np.zeros(6, dtype=bool)
    p = GB.pick_rule(P, np.array([3.0, 1.0, 1.0, 0.5, 0.5, 0.0]), S, none)
    assert (p["idx"], p["explore"], p["safe_idx"], p["target_idx"], p["target_lcb"]) == (1, 0, 1, -1, np.inf)
    p = GB.pick_rule(P, np.array([3.0, 1.0, 1.0, 1.0, 0.5, 0.0]), S, np.array([0, 0, 0, 1, 0, 0], dtype=bool))
    assert (p["idx"], p["explore"]) == (1, 0)           # l_S == l_T: the safe minimum (test_GoOSE.py:158-162)
    p = GB.pick_rule(P, np.array([3.0, 1.0, 1.0, 0.5, 0.5, 0.0]), S, T)
    assert (p["idx"], p["explore"], p["target_idx"], p["dist"]) == (2, 1, 3, 1.0)   # nearest safe point to z_3
    assert GB.pick_rule(P, np.zeros(6), none, T) is None


def test_safe_only_batch_when_the_target_is_empty():
    ds, P, beta, st, _ = _oracle_step("small0")
    picks = GB.goose_batch(P, ds, st["mean"][:, 0], st["var"][:, 0], beta, st["S"], np.zeros_like(st["S"]), 6)
    assert len(picks) == 6 and all(p["explore"] == 0 and p["target_idx"] == -1 for p in picks)
    assert len({p["idx"] for p in picks}) == 6


class _StubBatchBO:
    """Scripted GoOSE BO.Batch: pick 1 walks towards x = 0.3 (objective |x|^2 at 0.09 = f_opt) one iteration at a time."""

    def __init__(self):
        self.n_fun, self.nx_dim, self.it, self.added = 2, 2, 0, []
        self.plant_system = [lambda x, noise=0: float(np.sum(x * x)), lambda x, noise=0: 1.0 - float(np.sum(x * x))]

    def Batch(self, q):
        x0 = 0.1 * (self.it + 1)
        self.it += 1
        X = np.array([[x0 + 0.01 * k, 0.0] for k in range(q)])
        xt = np.full((q, 2), np.nan)
        xt[1:] = 0.5
        picks = [{"idx": k, "explore": int(k > 0), "safe_lcb": -1.0, "safe_idx": 0, "target_lcb": -2.0, "target_idx": 1, "dist": 0.1}
                 for k in range(q)]
        return X, np.full(q, -1.0), {"picks": picks, "chose": ["safe_minimum"] + ["explore"] * (q - 1), "x_target": xt,
                                     "min_safe_lcb": -1.0, "target_lcb": -2.0}

    def calculate_plant_outputs(self, x, noise=0):
        return np.array([p(x, noise) for p in self.plant_system])

    def add_sample(self, x, y, hypopt=None):
        self.added.append((np.asarray(x).copy(), np.asarray(y).copy(), hypopt))


def test_goose_batch_driver_adds_every_sample_and_stops_on_pick_one():
    import sbo_b200  # noqa: F401
    from sbo_b200 import drivers
    bo = _StubBatchBO()
    data = drivers.run_goose_batch(bo, 3, n_iteration=10, f_opt=0.09, tol=1e-9)
    # pick 1 is at x_0 = 0.1, 0.2, 0.3: the third iteration stops (|0.3^2 - 0.09| <= tol); pick 2 (0.31) would not
    assert len(data["info"]) == 3 and len(bo.added) == 9
    assert data["batch"] == [0, 0, 0, 1, 1, 1, 2, 2, 2] and data["i"] == list(range(9))
    assert np.allclose([a[0][0] for a in bo.added[:3]], [0.1, 0.11, 0.12])
    assert np.isnan(data["x_target_0"][0]) and data["x_target_0"][1] == 0.5 and data["obj"][1] == pytest.approx(0.0121)
    bo = _StubBatchBO()
    drivers.run_goose_batch(bo, 2, n_iteration=2, f_opt=None, hypopt="h")
    assert len(bo.added) == 4 and all(a[2] == "h" for a in bo.added)


def test_goose_batch_driver_stops_on_an_empty_safe_set():
    import sbo_b200  # noqa: F401
    from sbo_b200 import drivers

    class Empty(_StubBatchBO):
        def Batch(self, q):
            return np.zeros((0, 2)), np.zeros(0), {"picks": [], "chose": [], "x_target": np.zeros((0, 2)),
                                                   "min_safe_lcb": np.inf, "target_lcb": np.inf}

    with pytest.raises(drivers.EmptySafeSet):
        drivers.run_goose_batch(Empty(), 4)


def test_goose_batch_pick_layout_matches_the_header(tmp_path):
    """sbo_goose_batch_pick compiles as C99 and its ctypes mirror has the header's size and field offsets."""
    from sbo_b200 import _capi
    cls = _capi.GooseBatchPick
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "sbo_b200.h"', 'int main(void) {',
             '  printf("size %zu\\n", sizeof(sbo_goose_batch_pick));']
    lines += [f'  printf("{f} %zu\\n", offsetof(sbo_goose_batch_pick, {f}));' for f, _ in cls._fields_]
    lines += ['  return 0;', '}']
    src = tmp_path / "goose_batch_layout.c"
    src.write_text("\n".join(lines) + "\n")
    exe = tmp_path / "goose_batch_layout"
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    got = dict(ln.rsplit(" ", 1) for ln in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    assert int(got["size"]) == ctypes.sizeof(cls) == 56
    for f, _ in cls._fields_:
        assert int(got[f]) == getattr(cls, f).offset, f
