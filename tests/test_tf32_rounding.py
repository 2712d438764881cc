"""CPU: oracle.round_tf32, the NumPy emulation of PTX cvt.rna.tf32.f32 (round to 10 mantissa bits, nearest, ties away
from zero) that the GPU tests compare the TF32 and split-TF32 V rows with bit for bit.  Checked against an independent
FP64 statement of the same rounding and against hand-picked bit patterns."""
import numpy as np

from oracle.gp_oracle import round_tf32


def _tf32_ref(x):
    """Round float32 values to 11 significant bits, ties away from zero, in exact FP64 arithmetic (normal inputs)."""
    x = np.asarray(x, dtype=np.float32).astype(np.float64)
    _, e = np.frexp(x)                                  # |x| = f 2^e, f in [0.5, 1)
    ulp = np.ldexp(1.0, e - 11)
    return (np.sign(x) * np.floor(np.abs(x) / ulp + 0.5) * ulp).astype(np.float32)


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def test_ties_round_away_from_zero():
    # b + 2^-11 (b in [1, 2) with 10 mantissa bits) lies half-way between the TF32 neighbours b and b + 2^-10
    for b in (1.0, 1.5, 1.0 + 3 * 2.0 ** -10, 2.0 - 2.0 ** -10):
        for scale in (1.0, 2.0 ** 20, 2.0 ** -100, 2.0 ** 100):
            for sign in (1.0, -1.0):
                x = np.float32(sign * scale * (b + 2.0 ** -11))
                got = round_tf32(np.array([x]))[0]
                assert float(got) == sign * scale * (b + 2.0 ** -10), (x, got)     # away from zero
                assert got == _tf32_ref(np.array([x]))[0]


def test_nearest_below_and_above_the_tie():
    one = np.float32(1.0)
    step = np.float32(2.0 ** -23)
    half = np.float32(1.0 + 2.0 ** -11)
    just_below, just_above = np.float32(half - step), np.float32(half + step)
    assert round_tf32(np.array([just_below]))[0] == one
    assert round_tf32(np.array([just_above]))[0] == np.float32(1.0 + 2.0 ** -10)
    assert round_tf32(np.array([-just_below]))[0] == -one
    assert round_tf32(np.array([-just_above]))[0] == np.float32(-(1.0 + 2.0 ** -10))


def test_negative_values_mirror_positive_ones():
    x = np.random.default_rng(1).uniform(-1e3, 1e3, size=100000).astype(np.float32)
    assert np.array_equal(_bits(round_tf32(-x)), _bits(-round_tf32(x)))


def test_tf32_values_are_fixed_points():
    rng = np.random.default_rng(2)
    b = rng.integers(0, 2 ** 32, size=100000, dtype=np.uint64).astype(np.uint32) & np.uint32(0xFFFFE000)
    x = b.view(np.float32)
    x = x[np.isfinite(x) & ((b & np.uint32(0x7F800000)) != 0)]          # normal and finite TF32 patterns
    assert np.array_equal(_bits(round_tf32(x)), _bits(x))
    assert np.array_equal(_bits(round_tf32(np.float32([0.0, -0.0]))), _bits(np.float32([0.0, -0.0])))


def test_random_normal_values_match_the_exact_rounding():
    rng = np.random.default_rng(3)
    # magnitudes from 2^-120 to 2^120 (no subnormal inputs or results), both signs, plus V-row-like values in [-1, 1]
    x = (rng.choice([-1.0, 1.0], size=200000) * np.exp2(rng.uniform(-120, 120, size=200000))).astype(np.float32)
    y = rng.uniform(-1, 1, size=200000).astype(np.float32)
    y = y[np.abs(y) >= np.finfo(np.float32).tiny]
    for v in (x, y):
        got = round_tf32(v)
        assert np.array_equal(_bits(got), _bits(_tf32_ref(v)))
        assert np.all(_bits(got) & np.uint32(0x1FFF) == 0)                       # 13 low mantissa bits cleared
        assert np.all(np.abs(got.astype(np.float64) - v) <= np.abs(v.astype(np.float64)) * 2.0 ** -11)


def test_carry_into_the_next_binade():
    x = np.float32(np.nextafter(np.float32(2.0), np.float32(0.0)))          # 2 - 2^-23 rounds up to 2
    assert round_tf32(np.array([x]))[0] == np.float32(2.0)
    assert round_tf32(np.array([-x]))[0] == np.float32(-2.0)
