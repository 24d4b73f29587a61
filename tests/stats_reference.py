"""Exact summary statistics and ABC distances of a copy-number histogram, the error bounds of the f32 arithmetic
that computes them, and the histogram families on which both are checked.

TEST INFRASTRUCTURE, shared by test_stats_reference_host.py (the CPU oracle) and test_gpu_stats_reference.py (the
kernel's epilogue).  Nothing here calls the oracle or the library: the references are rationals (fractions) and
40-digit logarithms (mpmath), and the bounds follow from the sequence of f32 operations of ssa_kernel.cuh
(tile_stats, dynamics_take_warp, tile_ks, the ABC epilogue, entropy_term_q40, variance_from_moments), of capi.cu
target_stats and of the oracle's stats_from_dense / orc_ks_distance, which all perform the same operations.

u = 2^-24 is the unit roundoff of f32: a correctly rounded operation returns x (1 + e), |e| <= u.  Second-order
terms (u^2 against u) are covered by a factor (1 + 2^-20) on every bound.

  mean  = f32(s1) / f32(n), s1 = sum k c_k:    three roundings, relative error <= 3u.
  freq  = f32(n - c_0) / f32(n):               three roundings, relative error <= 3u.
  var   = f32(f64(n s2 - s1^2) / n / n):       the numerator is exact (128-bit integers); f64 rounds it and the two
                                               quotients by 2^-53 each, f32 rounds the result: relative error
                                               <= u + 3 * 2^-53.  It is 0 exactly when one class holds every cell.
  entropy = f32(sum_i floor(2^40 t_i)) 2^-40, t_i = -p_i log2 p_i computed by entropy_term_q40 from c_i and n:
    (A) p < 3/4: p^ = f32(c) / f32(n) = p (1 + th), |th| <= 3u.  ln p = e ln2 + ln f, f the mantissa of p^
        reduced to [sqrt(1/2), sqrt(2)], x = f - 1 exact.  The polynomial and its f32 evaluation:
        |lf - ln f| <= 1.3u |ln f| (1.27u measured on every f32 mantissa of that range); |ln f| <= |ln p|.  The
        two FMAs adding e (C1 + C2) round by u |ln p| each (the inner sum e C2 + lf is at most 1.001 |ln p|).  The
        argument error adds ln(1 + th), i.e. 3u / |ln p| relative.  Then p^ (3u), the product p^ ln p (u), the
        f32 constant log2(e) (0.23u) and the last product (u): t within (8.6 + 3 / |ln p|) u, taken as
        (10 + 3.01 / |ln p|) u; |ln p| >= ln(4/3) = 0.2877, so at most 20.5u.
    (B) p >= 3/4 (4c >= 3n, decided on the integers): x = -q, q = f32(n - c) / f32(n) = (1 - p)(1 + th'),
        |th'| <= 3u, goes to the polynomial directly (e = 0: the FMAs are exact), and p^ = f32(1 - q) is within
        2u of p.  d ln(1 + x) / dx = 1 / p <= 4/3 and |x| <= |ln(1 + x)|: 4u; polynomial 1.3u (1.16u measured
        over x in [-0.293, 0) at full f32 resolution); p^ 2u, products 2u, log2(e) 0.23u: t within 9.6u, taken
        as 12u.
    Truncation to 2^-40 loses less than 2^-40 per occupied class (m of them); the integer sum is exact; the
    final conversion rounds by u:
        |H^ - H| <= sum_i a(p_i) u t_i + u H + m 2^-40,   a(p) = max(12, 10 + 3.01 / |ln p|) below p = 3/4, 12 above,
    so in all cases |H^ - H| <= 21.5 u H + m 2^-40.
  KS    = max_k |f32(C_k) / f32(n) - f32(T_k) / f32(n_t)|: each CDF value within 3u relative (<= 3u absolute), the
          difference rounds by u: |KS^ - KS| <= 6u + u KS.
  relative distance d = |s - s_t| / s_t from statistics with absolute bounds b, b_t: the subtraction and the
          division round by u each, so |d^ - d| <= (b + b_t + u |s - s_t|) / (s_t - b_t) (1 + u)
                                                   + d b_t / (s_t - b_t) (1 + u) + u d.
"""
import math
from fractions import Fraction

import mpmath
import numpy as np

U = 2.0 ** -24
SLACK = 1.0 + 2.0 ** -20
Q40 = 2.0 ** -40


def as_dict(h):
    """{k: c} of the occupied classes of a dict or a dense array."""
    if isinstance(h, dict):
        return {int(k): int(c) for k, c in h.items() if c}
    a = np.asarray(h)
    return {int(k): int(a[k]) for k in np.flatnonzero(a)}


def dense(h, length=None):
    d = as_dict(h)
    out = np.zeros(max(length or 0, max(d, default=0) + 1), dtype=np.uint64)
    for k, c in d.items():
        out[k] = c
    return out


def _ent_term(c, n):
    p = mpmath.mpf(c) / n
    return -p * mpmath.log(p, 2)


def term_factor(p):
    """a(p): the error of one entropy term, in units of u t (derivation above)."""
    if p >= 0.75:
        return 12.0
    return max(12.0, 10.0 + 3.01 / abs(math.log(p)))


class Exact:
    """mean, frequency, variance (Fractions), entropy (mpmath, 40 digits) of a histogram, and the bounds."""

    def __init__(self, h):
        d = as_dict(h)
        self.d = d
        self.n = n = sum(d.values())
        self.m = len(d)
        self.kmax = max(d, default=0)
        if n == 0:
            self.mean = self.freq = self.var = Fraction(0)
            self.ent = mpmath.mpf(0)
            self.ent_err = 0.0
            return
        s1 = sum(k * c for k, c in d.items())
        s2 = sum(k * k * c for k, c in d.items())
        self.s1, self.s2 = s1, s2
        self.mean = Fraction(s1, n)
        self.freq = Fraction(n - d.get(0, 0), n)
        self.var = Fraction(n * s2 - s1 * s1, n * n)
        with mpmath.workdps(40):
            terms = [_ent_term(c, n) for c in d.values()]
            self.ent = mpmath.fsum(terms)
            self.ent_err = float(mpmath.fsum(term_factor(c / n) * t for c, t in zip(d.values(), terms)))

    # absolute error bounds of the f32 results
    def bound(self, stat):
        if stat == "mean":
            return SLACK * 3 * U * float(self.mean)
        if stat == "freq":
            return SLACK * 3 * U * float(self.freq)
        if stat == "var":
            return SLACK * U * float(self.var)
        if stat == "ent":
            return SLACK * (U * self.ent_err + U * float(self.ent)) + self.m * Q40
        raise KeyError(stat)

    def value(self, stat):
        return {"mean": self.mean, "freq": self.freq, "var": self.var, "ent": self.ent}[stat]


STATS = ("mean", "freq", "ent", "var")


def err_and_bound(ex, stat, got):
    """|got - exact| (exact arithmetic on the f32 value) and its bound."""
    v = ex.value(stat)
    if not np.isfinite(got):
        return math.inf, ex.bound(stat)
    if stat == "ent":
        with mpmath.workdps(40):
            err = float(abs(mpmath.mpf(float(got)) - v))
    else:
        err = float(abs(Fraction(float(got)) - v))
    return err, ex.bound(stat)


def ks_exact(h, t):
    """sup_k |F_h(k) - F_t(k)| over the two rational CDFs (zero-copy class included); 1 when either is empty."""
    a, b = as_dict(h), as_dict(t)
    na, nb = sum(a.values()), sum(b.values())
    if na == 0 or nb == 0:
        return Fraction(1)
    best, ca, cb = Fraction(0), 0, 0
    for k in sorted(set(a) | set(b)):  # (the CDFs only change at occupied classes)
        ca += a.get(k, 0)
        cb += b.get(k, 0)
        best = max(best, abs(Fraction(ca, na) - Fraction(cb, nb)))
    return best


def ks_bound(ks):
    return SLACK * U * (6 + float(ks))


def rel_exact(s, st):
    """|s - s_t| / s_t, exact (a Fraction or an mpf)."""
    return abs(s - st) / st


def rel_bound(s, st, b, bt):
    """Bound on |d^ - d| for d = |s - s_t| / s_t from statistics within b, b_t (derivation above)."""
    s, st = float(s), float(st)
    d = abs(s - st) / st
    den = st - bt
    assert den > 0, "the target statistic is not resolved by its own bound"
    return SLACK * ((b + bt + U * abs(s - st)) / den * (1 + U) + d * bt / den * (1 + U) + U * d)


# ------------------------------------------------------------------------------------------------------------
# histogram families: (name, {k: c}).  Every population is below 2^32 cells and every k below 2^16.
# ------------------------------------------------------------------------------------------------------------
def _window(kmax, step=3):
    h = {k: 1 + (7 * k) % 5 for k in range(0, kmax, step)}
    h[kmax] = 2
    return h


def families(seed=20261022, n_random=12):
    f = [
        # one class: variance and entropy exactly 0
        ("one_k0", {0: 5}), ("one_k1", {1: 1000}), ("one_k7_big", {7: 3_000_000_000}), ("one_k65534", {65534: 2 ** 20}),
        # a narrow spread at large k with one outlier
        ("narrow_1000", {1000: 999, 1001: 1}), ("narrow_20000", {20000: 39, 20001: 1}),
        ("narrow_2000_35", {2000: 3, 2001: 5}), ("narrow_65534", {65534: 100_000, 65533: 1}),
        ("narrow_65534_big", {65534: 2 ** 30, 65535: 1}), ("narrow_20000_wide", {19990: 7, 20000: 1_000_000, 20010: 7}),
        # near-degenerate populations: one class holds nearly every cell
        ("degen_1e7", {0: 9_999_999, 1: 1}), ("degen_2e31_5", {0: 2 ** 31 - 5, 7: 5}), ("degen_1000", {0: 999, 1: 1}),
        ("degen_2e31_1", {0: 2 ** 31 - 2, 255: 1}), ("degen_4e9_1000", {0: 4_000_000_000, 3: 1000}),
        ("degen_k_heavy", {5: 123_456_789, 0: 3}), ("degen_3cls", {0: 2 ** 30, 1: 1, 2: 1}),
        # n on either side of 2^24, where f32(n) starts to round
        ("n_2e24m1", {0: 2 ** 24 - 2, 3: 1}), ("n_2e24", {0: 2 ** 24 - 1, 3: 1}), ("n_2e24p1", {0: 2 ** 24, 3: 1}),
        ("n_2e24p3", {2: 2 ** 23 + 1, 5: 2 ** 23 + 2}), ("n_2e25p1", {1: 2 ** 25 - 7, 9: 8}),
        # s1 beyond 2^24, s2 beyond 2^53
        ("s1_big", {1000: 20_000, 3000: 5, 0: 11}), ("s2_big", {65000: 2 ** 22, 1: 3, 64000: 7}),
        ("s2_max", {65535: 2 ** 31, 0: 2 ** 31 - 1}),
        # every class occupied: entropy 16 bits, the largest number of terms
        ("all_uniform", {k: 1 for k in range(65536)}),
        ("all_mixed", {k: 1 + (k * 7919) % 13 for k in range(65536)}),
        # the window and stride edges of the strided k <= kmax loops
        ("kmax_127", _window(127)), ("kmax_128", _window(128)), ("kmax_255", _window(255)),
        ("kmax_256", _window(256)), ("kmax_511", _window(511)), ("kmax_512", _window(512)),
        ("kmax_127_only", {0: 3, 127: 2}), ("kmax_128_only", {0: 3, 128: 2}),
        ("kmax_511_only", {511: 1, 1: 1}), ("kmax_512_only", {512: 1, 1: 1}),
    ]
    rng = np.random.default_rng(seed)
    for i in range(n_random):
        kmax = int(rng.choice([31, 200, 511, 3000, 40000]))
        occ = rng.choice(kmax + 1, size=int(rng.integers(1, min(kmax + 1, 400) + 1)), replace=False)
        counts = np.exp(rng.uniform(0, math.log(1e6), occ.size)).astype(np.int64) + 1
        f.append((f"random_{i}", {int(k): int(c) for k, c in zip(occ, counts)}))
    return f


# ABC targets: a bulk, a narrow, a near-degenerate one, and one that is far out
TARGETS = {
    "bulk": {0: 400, 1: 120, 2: 90, 3: 60, 5: 40, 9: 20, 30: 5},
    "narrow_1000": {1000: 999, 1001: 1},
    "degen": {0: 9_999_999, 1: 1},
    "far": {40000: 3, 40001: 2},
}
