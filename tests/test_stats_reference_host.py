"""The CPU oracle's summary statistics (stats_from_dense through orc_stats) and KS distance (orc_ks_distance)
against exact references, within the error bounds derived in stats_reference.py.

The kernel's epilogue repeats the oracle's operations bit for bit (test_gpu_parity.py), so these bounds hold for
what the library reports too; test_gpu_stats_reference.py checks that on the GPU, path by path.
"""
import math
from fractions import Fraction

import numpy as np
import pytest

import oracle_binding as ob
import stats_reference as sr

FAMILIES = sr.families()
_EXACT = {}


def exact(name, h):
    if name not in _EXACT:
        _EXACT[name] = sr.Exact(h)
    return _EXACT[name]


@pytest.mark.parametrize("name,h", FAMILIES, ids=[n for n, _ in FAMILIES])
def test_oracle_stats_within_bounds(name, h):
    ex = exact(name, h)
    got = dict(zip(("mean", "freq", "ent", "var"), ob.stats(sr.dense(h))))
    for stat in sr.STATS:
        err, bound = sr.err_and_bound(ex, stat, got[stat])
        assert err <= bound, f"{name} {stat}: {got[stat]!r} vs exact {float(ex.value(stat))!r}: error {err:.3g} > bound {bound:.3g}"
    # variance and entropy are exactly 0 for one class and only then; the variance is never negative
    assert (got["var"] == 0) == (ex.m == 1) and got["var"] >= 0
    assert (got["ent"] == 0) == (ex.m == 1)


def test_cancellation_and_degenerate_cases():
    """Histograms on which f32(s2)/n - mu^2 cancels (it gives -32 and 0 on the first two) and on which rounding
    p = c/n before its log loses a near-degenerate population's entropy (by percent)."""
    m, f, e, v = ob.stats(sr.dense({20000: 39, 20001: 1}))
    assert abs(v - 0.024375) <= 2 * sr.U * 0.024375
    m, f, e, v = ob.stats(sr.dense({2000: 3, 2001: 5}))
    assert v == np.float32(0.234375)  # (15/64: exact in f32, and the result is correctly rounded)
    m, f, e, v = ob.stats(sr.dense({1000: 999, 1001: 1}))
    assert abs(v - 0.000999) <= 2 * sr.U * 0.000999
    for h in ({0: 9_999_999, 1: 1}, {0: 2 ** 31 - 5, 7: 5}):
        ex = sr.Exact(h)
        e = ob.stats(sr.dense(h))[2]
        assert abs(e - float(ex.ent)) <= 21.5 * sr.U * float(ex.ent) + ex.m * sr.Q40


def test_extinct_population():
    assert ob.stats(np.zeros(8, dtype=np.uint64)) == (0.0, 0.0, 0.0, 0.0)
    assert ob.ks_distance(np.zeros(8, dtype=np.uint64), sr.dense({0: 3, 2: 1})) == 1.0
    assert ob.ks_distance(sr.dense({0: 3, 2: 1}), np.zeros(4, dtype=np.uint64)) == 1.0


KS_PAIRS = [(n, t) for n, _ in FAMILIES[::3] for t in sr.TARGETS] + [
    ("narrow_1000", "narrow_1000"), ("degen_1e7", "degen")]


@pytest.mark.parametrize("name,target", KS_PAIRS, ids=[f"{n}-{t}" for n, t in KS_PAIRS])
def test_oracle_ks_within_bound(name, target):
    h = dict(FAMILIES)[name]
    t = sr.TARGETS[target]
    got = ob.ks_distance(sr.dense(h), sr.dense(t))
    ks = sr.ks_exact(h, t)
    err = float(abs(Fraction(float(got)) - ks))
    assert err <= sr.ks_bound(ks), (got, float(ks), err)
    # and in either order, on histograms padded to different lengths (the CDF past a histogram's end is 1)
    got2 = ob.ks_distance(sr.dense(t, 70000), sr.dense(h))
    assert float(abs(Fraction(float(got2)) - ks)) <= sr.ks_bound(ks)


def test_ks_exact_reference_sanity():
    """The rational reference itself: identical histograms 0, disjoint ones 1, a hand-computed case."""
    assert sr.ks_exact({3: 2, 5: 1}, {3: 4, 5: 2}) == 0
    assert sr.ks_exact({0: 5}, {9: 1}) == 1
    assert sr.ks_exact({0: 1, 2: 1}, {1: 1}) == Fraction(1, 2)
    assert sr.ks_exact({}, {1: 1}) == 1


def test_entropy_bound_is_tight_enough():
    """The entropy bound is not so loose that it would pass the former p-rounding error: on {0: 10^7 - 1, 1: 1}
    that error is 1.1 % of H, the bound below 2.5e-6 of it."""
    ex = sr.Exact({0: 9_999_999, 1: 1})
    assert ex.bound("ent") < 2.5e-6 * float(ex.ent)
    # the entropy reference: two classes, closed form
    p = 1e-7
    assert math.isclose(float(ex.ent), -(p * math.log2(p) + (1 - p) * math.log1p(-p) / math.log(2)), rel_tol=1e-12)


def test_report_worst_ratios():
    """The largest observed / bound ratio per statistic over every family (printed with -s)."""
    worst = {s: 0.0 for s in sr.STATS}
    for name, h in FAMILIES:
        ex = exact(name, h)
        got = dict(zip(("mean", "freq", "ent", "var"), ob.stats(sr.dense(h))))
        for s in sr.STATS:
            err, bound = sr.err_and_bound(ex, s, got[s])
            if bound > 0:
                worst[s] = max(worst[s], err / bound)
    print("\noracle observed/bound:", {s: round(v, 4) for s, v in worst.items()})
    assert all(v <= 1.0 for v in worst.values())
