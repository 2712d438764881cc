"""CPU: the NumPy reference of the fantasy GoOSE target (tests/goose_fantasy_ref.py) against the oracle's fantasy
quantities -- brute-force augmented inference per (x, z), and the expander counts of the same pairs."""
import numpy as np

from conftest import golden_ds
from goose_fantasy_ref import fantasy_target_blocks, goose_step_fantasy, goose_target_fantasy


def _case(oracle, c3, n=20, ppd=14, beta=2.0, rule="any"):
    ds = golden_ds(oracle, c3, n)
    pts = oracle.make_grid(c3["lo"], c3["hi"], [ppd, ppd])
    mean, var = oracle.posterior_chol(pts, ds)
    lcb, _ = oracle.bounds(mean, var, beta)
    return ds, pts, beta, lcb, oracle.safe_mask(lcb), oracle.unsafe_mask(lcb, rule)


def test_target_agrees_with_augmented_inference(oracle, c3):
    ds, pts, beta, lcb, S, Z = _case(oracle, c3, ppd=10)
    xs, zs = np.flatnonzero(S), np.flatnonzero(Z)
    assert xs.size and zs.size
    tg = goose_target_fantasy(pts, ds, beta, S, Z, lcb)
    bf = np.full(zs.size, -np.inf)                     # best over x of min_i lcb'_i(z | x), normalised units
    for x in xs:
        lcb_aug = oracle.fantasy_by_augmentation(pts[x], pts[zs], ds, beta)[:, 1:]
        bf = np.maximum(bf, np.min(lcb_aug / ds["Y_std"][1:], axis=1))
    clear = np.abs(bf) > 1e-6                          # the two forms agree to ~1e-7 (test_rank1_fantasy_vs_augmented_inference)
    assert clear.sum() >= zs.size - 2
    assert np.array_equal(tg["mask"][zs][clear], (bf >= 0)[clear])
    assert tg["mask"].sum() > 0 and not tg["mask"][~Z].any()
    np.testing.assert_allclose(tg["best_margin"][zs], bf, rtol=1e-6, atol=1e-7)


def test_target_is_the_column_or_of_the_counts(oracle, c3):
    for n, beta, rule in ((20, 2.0, "any"), (5, 3.0, "all"), (35, 2.0, "all")):
        ds, pts, beta, lcb, S, Z = _case(oracle, c3, n=n, beta=beta, rule=rule)
        counts = oracle.fantasy_counts(pts, ds, beta, S, Z)
        T, _ = fantasy_target_blocks(pts, ds, beta, S, Z)
        assert (T.sum() == 0) == (counts.sum() == 0)
        assert T.sum() <= counts.sum() and T.sum() <= Z.sum()
        assert not T[~Z].any()


def test_empty_target(oracle, c1):
    ds = golden_ds(oracle, c1, 4)
    pts = oracle.make_grid([5.0, 5.0], [6.0, 6.0], [8, 8])      # far from the data: nothing is safe
    st = goose_step_fantasy(pts, ds, 3.0)
    assert st["target_idx"] == -1 and st["target_lcb"] == np.inf and not st["target_mask"].any()
    assert st["x_new_idx"] == st["safe_min_idx"] == -1
    counts = oracle.fantasy_counts(pts, ds, 3.0, st["S"], st["Z"])
    assert counts.sum() == 0


def test_step_decision_rule(oracle, c3):
    ds = golden_ds(oracle, c3, 20)
    pts = oracle.make_grid(c3["lo"], c3["hi"], [14, 14])
    st = goose_step_fantasy(pts, ds, 2.0, "any")
    assert st["target_idx"] >= 0 and st["target_mask"][st["target_idx"]]
    if st["safe_min_lcb"] <= st["target_lcb"]:
        assert st["x_new_idx"] == st["safe_min_idx"] and st["explore_idx"] == -1
    else:
        assert st["S"][st["x_new_idx"]] and st["explore_idx"] == st["x_new_idx"]
