"""CPU: the batch SafeOpt acquisition's math and host logic -- the incremental variance downdate against brute-force
augmentation for every covariance function, the pick rule on hand-made masks, the batch driver loop with a stub BO, and the
C layout of sbo_batch_pick against its ctypes mirror."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import matern_ref as MR
import safeopt_batch_ref as B
from conftest import ROOT


def _small():
    from sbo_b200 import workloads
    ds, lo, hi, pts, beta = workloads.small(d=3, pts_per_dim=9, n=30, seed=11, G=2)
    from oracle import gp_oracle as O
    return ds, O.make_grid(lo, hi, pts)


@pytest.mark.parametrize("kernel", MR.KERNELS)
def test_incremental_downdate_equals_bruteforce_augmentation(kernel):
    ds, P = _small()
    _, var = MR.posterior_chol(P, ds, kernel)
    ys2 = ds["Y_std"][0] ** 2
    sf2 = float(np.exp(2.0 * ds["hypopt"][3, 0]))
    picks = [100, 7, 500, 100, 631, 8]                  # 100 twice: a repeated pick is an ordinary observation
    dd = B.Downdate(P, ds, var[:, 0], kernel)
    for b in range(len(picks)):
        dd.commit(P[picks[b]])
        ref = B.variance_bruteforce(P, ds, P[picks[:b + 1]], kernel)
        assert np.max(np.abs(dd.v - ref)) / ys2 <= 1e-12 * sf2, (kernel, b)
    assert dd.v[100] < var[100, 0] and np.all(dd.v <= var[:, 0])


def test_pick_rule_ties_and_empty_sets():
    v = np.array([1.0, 4.0, 4.0, 9.0, 9.0, 0.25])
    M = np.array([1, 1, 1, 0, 0, 0], dtype=bool)
    E = np.array([0, 0, 0, 1, 1, 1], dtype=bool)
    p = B.pick_rule(v, M, E)
    assert (p["idx_min"], p["idx_exp"]) == (1, 3)          # lowest index on ties inside each set
    assert p["std_min"] == 2.0 and p["std_exp"] == 3.0
    assert (p["idx"], p["from_expander"]) == (3, 1)
    p = B.pick_rule(np.array([9.0, 4.0, 9.0, 9.0, 9.0, 1.0]), M, E)
    assert (p["idx"], p["from_expander"]) == (3, 1)        # std_M == std_E: not greater -> E (test_SafeOpt.py:153-158)
    p = B.pick_rule(np.array([16.0, 4.0, 9.0, 9.0, 9.0, 1.0]), M, E)
    assert (p["idx"], p["from_expander"]) == (0, 0)
    none = np.zeros(6, dtype=bool)
    p = B.pick_rule(v, none, E)
    assert (p["idx"], p["from_expander"], p["idx_min"], p["std_min"]) == (3, 1, -1, 0.0)
    p = B.pick_rule(np.zeros(6), M, none)                   # E empty: M's point even at std 0
    assert (p["idx"], p["from_expander"], p["idx_exp"], p["std_exp"]) == (0, 0, -1, 0.0)
    assert B.pick_rule(v, none, none) is None


def test_single_candidate_is_picked_again_and_both_empty_stops():
    ds, P = _small()
    _, var = MR.posterior_chol(P, ds, "RBF")
    M = np.zeros(P.shape[0], dtype=bool)
    M[42] = True
    picks = B.safeopt_batch(P, ds, var[:, 0], M, np.zeros_like(M), 4)
    assert [p["idx"] for p in picks] == [42] * 4
    s = [p["std_min"] for p in picks]
    assert s[0] == pytest.approx(np.sqrt(var[42, 0]), rel=1e-15) and s[0] > s[1] > s[2] > s[3] > 0
    assert B.safeopt_batch(P, ds, var[:, 0], np.zeros_like(M), np.zeros_like(M), 4) == []


def test_batch_spreads_out_over_the_candidates():
    ds, P = _small()
    _, var = MR.posterior_chol(P, ds, "Matern52")
    M = np.zeros(P.shape[0], dtype=bool)
    E = np.zeros_like(M)
    M[::7] = True
    E[3::11] = True
    picks = B.safeopt_batch(P, ds, var[:, 0], M, E, 6, kernel="Matern52", rtol=1e-9)
    assert len(picks) == 6 and len({p["idx"] for p in picks}) == 6
    assert picks[0]["idx"] == (B.pick_rule(var[:, 0], M, E))["idx"]
    for p in picks:
        assert (M if p["from_expander"] == 0 else E)[p["idx"]]


class _StubBatchBO:
    """Scripted BO.Batch: picks' stds shrink by half per iteration; records the samples it is given."""

    def __init__(self, q_max=3):
        self.n_fun, self.nx_dim, self.it, self.added = 2, 2, 0, []

    def Batch(self, q):
        s = 0.5 ** self.it
        self.it += 1
        X = np.array([[0.1 * k, -0.1 * k] for k in range(q)])
        picks = [{"idx": k, "from_expander": k % 2, "std_min": s, "idx_min": 0, "std_exp": s / 2, "idx_exp": 1} for k in range(q)]
        return X, np.full(q, s), {"picks": picks, "chose": ["minimizer"] * q, "std_minimizer": s, "std_expander": s / 2}

    def calculate_plant_outputs(self, x, noise=0):
        return np.array([float(np.sum(x * x)), 1.0 - float(np.sum(x * x))])

    def add_sample(self, x, y, hypopt=None):
        self.added.append((np.asarray(x).copy(), np.asarray(y).copy(), hypopt))


def test_batch_driver_adds_every_sample_and_stops_on_pick_one():
    import sbo_b200  # noqa: F401
    from sbo_b200 import drivers
    bo = _StubBatchBO()
    data = drivers.run_safeopt_batch(bo, 3, n_iteration=10, stop_std=0.2)
    # stds of pick 1: 1, 0.5, 0.25, 0.125 -> the 4th iteration stops (both below 0.2)
    assert len(data["info"]) == 4 and len(bo.added) == 12
    assert data["batch"] == [0, 0, 0, 1, 1, 1, 2, 2, 2, 3, 3, 3] and data["i"] == list(range(12))
    assert np.allclose([a[0] for a in bo.added[:3]], [[0.0, 0.0], [0.1, -0.1], [0.2, -0.2]])
    assert data["x_1"][1] == pytest.approx(-0.1) and data["obj"][2] == pytest.approx(0.08)
    bo = _StubBatchBO()
    drivers.run_safeopt_batch(bo, 2, n_iteration=2, stop_std=0.0, hypopt="h")
    assert len(bo.added) == 4 and all(a[2] == "h" for a in bo.added)


def test_batch_driver_stops_on_an_empty_safe_set():
    import sbo_b200  # noqa: F401
    from sbo_b200 import drivers

    class Empty(_StubBatchBO):
        def Batch(self, q):
            return np.zeros((0, 2)), np.zeros(0), {"picks": [], "chose": [], "std_minimizer": 0.0, "std_expander": 0.0}

    with pytest.raises(drivers.EmptySafeSet):
        drivers.run_safeopt_batch(Empty(), 4)


def test_batch_pick_layout_matches_the_header(tmp_path):
    """sbo_batch_pick compiles as C99 and its ctypes mirror has the header's size and field offsets."""
    from sbo_b200 import _capi
    cls = _capi.BatchPick
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "sbo_b200.h"', 'int main(void) {',
             '  printf("size %zu\\n", sizeof(sbo_batch_pick));']
    lines += [f'  printf("{f} %zu\\n", offsetof(sbo_batch_pick, {f}));' for f, _ in cls._fields_]
    lines += ['  printf("SBO_BATCH_MAX_Q %d\\n", SBO_BATCH_MAX_Q);', '  return 0;', '}']
    src = tmp_path / "batch_layout.c"
    src.write_text("\n".join(lines) + "\n")
    exe = tmp_path / "batch_layout"
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    got = dict(ln.rsplit(" ", 1) for ln in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    assert int(got["size"]) == ctypes.sizeof(cls) == 48
    for f, _ in cls._fields_:
        assert int(got[f]) == getattr(cls, f).offset, f
    assert int(got["SBO_BATCH_MAX_Q"]) == _capi.BATCH_MAX_Q
