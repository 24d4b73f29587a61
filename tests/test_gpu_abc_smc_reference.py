"""ABC-SMC (DESIGN.md section 9) against references that do not restate the kernels' formulas: a vectorised numpy
Philox4x32-10, the prior draws rounded exactly, the proposals against scipy's truncated normal, the importance-sampling
identity on the prior box, the weight kernel against float64 within an error bound derived from its arithmetic, and a
Python replay of the driver that must give the result of ecdna_b200_abc_smc byte for byte.

Only the tests marked gpu need a device; the Philox and exact-rounding references are checked on the CPU."""
import math
from fractions import Fraction

import numpy as np
import pytest
from scipy import special, stats

import oracle_binding as ob
from test_gpu_abc_smc import BINS, BOX, DOMAIN, UINT64_MAX, _rho
from test_gpu_parity import oracle_opts

RANGES = [BOX["b1_range"], BOX["d0_range"], BOX["d1_range"]]
PRIOR_DOMAIN = (0xABC0ABC0, 0xFFFFFFFF)  # counter words 0 and 1 of the prior draws (capi.cu prior_kernel)
U32 = 2.0 ** -24  # unit roundoff of f32
U64 = 2.0 ** -53


# ---------------------------------------------------------------------------------------------------------------
# 0. Philox4x32-10 in numpy, and the uniforms built on it
# ---------------------------------------------------------------------------------------------------------------
def philox(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 (Random123) on arrays of counter words: returns the four output words as uint64 arrays."""
    mask = np.uint64(0xFFFFFFFF)
    c = [np.asarray(x, dtype=np.uint64) & mask for x in (c0, c1, c2, c3)]
    c = np.broadcast_arrays(*c)
    c0, c1, c2, c3 = (x.copy() for x in c)
    k0, k1 = np.uint64(k0) & mask, np.uint64(k1) & mask
    for r in range(10):
        p0, p1 = np.uint64(0xD2511F53) * c0, np.uint64(0xCD9E8D57) * c2  # 32 x 32 bits: exact in 64
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & mask, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & mask
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & mask, (k1 + np.uint64(0xBB67AE85)) & mask
    return c0, c1, c2, c3


def u53(a, b):
    """u in [0, 1) from 53 bits of two words (abc_smc.cu u53, numpy's random_sample construction)."""
    return ((a >> np.uint64(5)).astype(np.float64) * 67108864.0 + (b >> np.uint64(6)).astype(np.float64)) * 2.0 ** -53


def u24(a):
    """u in [0, 1) from the top 24 bits of one word, in f32 (capi.cu prior_kernel)."""
    return ((a >> np.uint64(8)).astype(np.float32) * np.float32(U32)).astype(np.float32)


def _idx_words(idx):
    idx = np.asarray(idx, dtype=np.uint64)
    return idx & np.uint64(0xFFFFFFFF), idx >> np.uint64(32)


def proposal_uniforms(seed, idx):
    """The four 53-bit uniforms of draw idx's proposal: parent, b1, d0, d1."""
    lo, hi = _idx_words(idx)
    x = philox(DOMAIN, 0, lo, hi, seed & 0xFFFFFFFF, seed >> 32)
    y = philox(DOMAIN, 1, lo, hi, seed & 0xFFFFFFFF, seed >> 32)
    return np.stack([u53(x[0], x[1]), u53(x[2], x[3]), u53(y[0], y[1]), u53(y[2], y[3])], axis=1)


def fma_f32(u, d, lo):
    """f32(u * d + lo) rounded once, as an f32 fma: u * d is exact in f64 (24 x 24 bits), the sum is rounded to f64
    with its error kept (TwoSum), and the one case where rounding that f64 to f32 differs from rounding the exact sum
    (the f64 sum exactly halfway between two f32 values, with a non-zero error) is settled by the error's sign."""
    p = np.asarray(u, dtype=np.float32).astype(np.float64) * np.asarray(d, dtype=np.float32).astype(np.float64)
    l = np.broadcast_to(np.asarray(lo, dtype=np.float32).astype(np.float64), p.shape)
    s = p + l
    bp = s - l
    e = (p - bp) + (l - (s - bp))
    r = s.astype(np.float32)
    rd = r.astype(np.float64)
    other = np.nextafter(r, np.where(s > rd, np.float32(np.inf), np.float32(-np.inf)))
    tie = (s != rd) & (s == (rd + other.astype(np.float64)) * 0.5) & (e != 0)
    return np.where(tie, np.where(e > 0, np.maximum(r, other), np.minimum(r, other)), r).astype(np.float32)


def prior_reference(seed, idx_begin, n, b0, ranges):
    lo, hi = _idx_words(np.arange(n, dtype=np.uint64) + np.uint64(idx_begin))
    x = philox(PRIOR_DOMAIN[0], PRIOR_DOMAIN[1], lo, hi, seed & 0xFFFFFFFF, seed >> 32)
    out = np.zeros((n, 4), dtype=np.float32)
    out[:, 0] = np.float32(b0)
    for k, (a, b) in enumerate(ranges):
        a, b = np.float32(a), np.float32(b)
        out[:, k + 1] = fma_f32(u24(x[k]), b - a, a)  # (hi - lo: one f32 subtraction, as in the kernel)
    return out


def _rn32(x):
    """Round a Fraction to the nearest f32, ties to even."""
    f = np.float32(float(x))
    cands = [np.nextafter(f, np.float32(-np.inf)), f, np.nextafter(f, np.float32(np.inf))]
    best = min(cands, key=lambda c: (abs(Fraction(float(c)) - x), int(np.array(c).view(np.uint32)) & 1))
    return np.float32(best)


KAT = [([0, 0, 0, 0], [0, 0], [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]),
       ([0xFFFFFFFF] * 4, [0xFFFFFFFF] * 2, [0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD]),
       ([0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344], [0xA4093822, 0x299F31D0],
        [0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1])]  # Random123 kat_vectors (as in test_oracle_kat.py)


def test_numpy_philox_matches_random123_and_the_oracle():
    for ctr, key, want in KAT:
        assert [int(w[()]) for w in philox(*ctr, *key)] == want
    rng = np.random.default_rng(1)
    ctr = rng.integers(0, 2**32, (4000, 4), dtype=np.uint64)
    key = rng.integers(0, 2**32, (4000, 2), dtype=np.uint64)
    ctr[:1000, 2:] |= np.uint64(0x80000000)  # counter words >= 2^31 (the high index word of draws past 2^63)
    ctr[1000:1100] = 0xFFFFFFFF
    got = np.stack(philox(ctr[:, 0], ctr[:, 1], ctr[:, 2], ctr[:, 3], 0, 0), axis=1)  # key 0 in bulk ...
    for i in range(0, 4000, 7):
        np.testing.assert_array_equal(got[i], ob.philox(ctr[i], [0, 0]))
    for i in range(0, 4000, 13):  # ... and per row with a random key
        one = np.array([int(w[()]) for w in philox(*ctr[i], *key[i])])
        np.testing.assert_array_equal(one, ob.philox(ctr[i], key[i]))
    # the uniforms: u53 in [0, 1) with its extremes, u24 exact multiples of 2^-24
    top = np.array([0xFFFFFFFF], dtype=np.uint64)
    assert u53(top, top)[0] == 1.0 - 2.0 ** -53 and u53(top * 0, top * 0)[0] == 0.0
    assert u24(top)[0] == np.float32(1.0 - 2.0 ** -24) and u24(np.array([255], dtype=np.uint64))[0] == 0.0
    u = proposal_uniforms(26, np.array([5, 2**32 + 5], dtype=np.uint64))
    assert u.shape == (2, 4) and not np.array_equal(u[0], u[1])  # the high index word enters the counter


def test_exact_fma_reference_against_fractions():
    """fma_f32 is the correctly rounded u * d + lo, including the halfway cases where f64 double rounding fails."""
    rng = np.random.default_rng(2)
    n = 3000
    u = (rng.integers(0, 2**24, n) * U32).astype(np.float32)
    lo = rng.uniform(0, 3, n).astype(np.float32)
    d = (rng.uniform(0, 3, n).astype(np.float32) - lo).astype(np.float32)
    # halfway cases: 6700417 * 641 = 2^32 + 1 and 65537 * 65535 = 2^32 - 1, so u * d = 2^-24 +- 2^-56; the f64 sum
    # with lo = 1 (+ 2^-23) lands exactly between two f32 values and the 2^-56 decides
    u[:2], d[:2], lo[:2] = np.float32(6700417 * U32), np.float32(641 * 2.0 ** -32), np.float32(1.0)
    u[2:4], d[2:4], lo[2:4] = np.float32(65537 * U32), np.float32(65535 * 2.0 ** -32), np.float32(1.0 + 2.0 ** -23)
    got = fma_f32(u, d, lo)
    exact = [_rn32(Fraction(float(a)) * Fraction(float(b)) + Fraction(float(c))) for a, b, c in zip(u, d, lo)]
    np.testing.assert_array_equal(got.view(np.uint32), np.array(exact, dtype=np.float32).view(np.uint32))
    naive = (u.astype(np.float64) * d.astype(np.float64) + lo.astype(np.float64)).astype(np.float32)
    assert np.any(naive != got), "no halfway case exercised"


# ---------------------------------------------------------------------------------------------------------------
# 1. prior draws
# ---------------------------------------------------------------------------------------------------------------
PRIOR_BOX = [(1.0, 2.0), (0.0, 0.5), (0.1, 0.7)]


@pytest.mark.gpu
@pytest.mark.parametrize("idx_begin, n", [(2**32 - 1000, 2000), (2**32 - 1, 1), (0, 1), (77, 1000), (2**40 + 3, 4097)])
def test_prior_draws_bit_for_bit(ctx, idx_begin, n):
    for seed, ranges in ((26, PRIOR_BOX), (2**40 + 9, [(0.3, 3.7), (0.25, 0.25), (0.0, 1e-3)])):
        got = ctx.abc_draw_priors(seed, idx_begin, n, 1.25, *ranges)
        ref = prior_reference(seed, idx_begin, n, 1.25, ranges)
        np.testing.assert_array_equal(got.view(np.uint32), ref.view(np.uint32))


@pytest.mark.gpu
def test_prior_draws_are_uniform(ctx):
    n = 1_000_000
    ranges = [(1.0, 2.0), (0.0, 0.5), (0.2, 0.2)]
    got = ctx.abc_draw_priors(7, 2**32 - n // 2, n, 1.0, *ranges)
    assert np.all(got[:, 0] == 1.0)
    for k, (lo, hi) in enumerate(ranges):
        x = got[:, k + 1]
        assert np.all((x >= np.float32(lo)) & (x <= np.float32(hi)))
        if lo == hi:
            assert np.all(x == np.float32(lo))
            continue
        p = stats.kstest(x.astype(np.float64), stats.uniform(lo, hi - lo).cdf).pvalue
        assert p > 1e-3, (k, p)


# ---------------------------------------------------------------------------------------------------------------
# 2. proposals
# ---------------------------------------------------------------------------------------------------------------
def _truncnorm(lo, hi, parent, sigma):
    lo, hi, c = float(np.float32(lo)), float(np.float32(hi)), float(np.float32(parent))
    return stats.truncnorm((lo - c) / sigma, (hi - c) / sigma, loc=c, scale=sigma)


SINGLE = {  # (parent b1, d0, d1), sigma, box: every case of the truncation on one parent
    "lo-edges": ((1.0, 0.0, 0.25), (0.2, 0.1, 10.0), BOX),  # b1 on lo, d0 exactly 0, d1 with sigma >> width
    "hi-edge": ((2.0, 0.25, 0.3), (0.5, 0.01, 0.0), BOX),   # b1 on hi, d0 sigma << width, d1 sigma = 0 (a copy)
    "fixed": ((1.5, 0.5, 0.2), (0.3, 0.2, 0.1), dict(BOX, d1_range=(0.2, 0.2))),  # d0 on hi, d1 lo == hi
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(SINGLE))
def test_proposal_single_parent_is_truncated_normal(ctx, case):
    parent, sigma, box = SINGLE[case]
    prev = np.array([[1.0, *parent]], dtype=np.float32)
    n = 1_000_000
    rates, par = ctx.abc_smc_propose(5, 2**32 - 3000, n, prev, np.array([1.0]), sigma, **box)
    assert np.all(par == 0) and np.all(rates[:, 0] == 1.0)
    ranges = [box["b1_range"], box["d0_range"], box["d1_range"]]
    for k in range(3):
        lo, hi = ranges[k]
        x = rates[:, k + 1]
        assert np.all((x >= np.float32(lo)) & (x <= np.float32(hi))), k
        if lo == hi or sigma[k] == 0:
            assert np.all(x.view(np.uint32) == prev[0, k + 1].view(np.uint32)), k  # an exact copy of the parent
            continue
        p = stats.kstest(x.astype(np.float64), _truncnorm(lo, hi, parent[k], sigma[k]).cdf).pvalue
        assert p > 1e-3, (case, k, p)


@pytest.mark.gpu
def test_proposal_parent_counts_follow_the_weights(ctx):
    rng = np.random.default_rng(4)
    M, n = 50, 1_000_000
    prev = np.column_stack([np.ones(M), rng.uniform(1, 2, M), rng.uniform(0, 0.5, (M, 2))]).astype(np.float32)
    W = rng.uniform(0, 1, M) ** 3
    W[17] = 0.0
    W /= W.sum()
    _, par = ctx.abc_smc_propose(8, 1000, n, prev, np.cumsum(W), (0.1, 0.1, 0.1), **BOX)
    counts = np.bincount(par, minlength=M)
    assert len(counts) == M and counts[17] == 0
    keep = W > 0
    p = stats.chisquare(counts[keep], n * W[keep]).pvalue
    assert p > 1e-3, p


def _edge_population(rng, M):
    """Parents crowded against d0 = 0 and the (b1 = 1, d1 = 0) corner, a third spread over the box."""
    b1, d0, d1 = rng.uniform(1, 2, M), rng.uniform(0, 0.5, M), rng.uniform(0, 0.5, M)
    a, b = M // 3, 2 * M // 3
    d0[:a] = rng.uniform(0, 0.02, a)
    d0[:a:3] = 0.0
    b1[a:b], d1[a:b] = 1.0 + rng.uniform(0, 0.03, b - a), rng.uniform(0, 0.015, b - a)
    b1[a:b:4], d1[a:b:4] = 1.0, 0.0
    return np.column_stack([np.ones(M), b1, d0, d1]).astype(np.float32)


@pytest.mark.gpu
def test_proposal_mixture_marginal_within_dkw_band(ctx):
    rng = np.random.default_rng(5)
    M, n = 500, 1_000_000
    prev = _edge_population(rng, M)
    W = rng.uniform(0.1, 1.0, M)
    W /= W.sum()
    sigma = (0.15, 0.06, 0.04)
    rates, _ = ctx.abc_smc_propose(9, 2**33, n, prev, np.cumsum(W), sigma, **BOX)
    band = math.sqrt(math.log(2 / 1e-6) / (2 * n))  # DKW: P(sup |F_n - F| > band) <= 1e-6
    for k, (lo, hi) in enumerate(RANGES):
        grid = np.linspace(lo, hi, 2000)
        c = prev[:, k + 1].astype(np.float64)[:, None]
        a, b = special.ndtr((lo - c) / sigma[k]), special.ndtr((hi - c) / sigma[k])
        F = W @ np.clip((special.ndtr((grid[None, :] - c) / sigma[k]) - a) / (b - a), 0, 1)
        emp = np.searchsorted(np.sort(rates[:, k + 1].astype(np.float64)), grid, side="right") / n
        dev = np.max(np.abs(emp - F))
        assert dev < band, (k, dev, band)


@pytest.mark.gpu
def test_proposal_index_handling(ctx):
    rng = np.random.default_rng(6)
    M, n, seed, idx0 = 40, 1000, 2**33 + 17, 2**32 - 100
    prev = np.column_stack([np.ones(M), rng.uniform(1, 2, M), rng.uniform(0, 0.5, M), np.full(M, 0.2)]).astype(np.float32)
    W = rng.uniform(0.1, 1, M)
    cum = np.cumsum(W / W.sum())
    sigma = (0.2, 0.05, 0.1)
    box = dict(BOX, d1_range=(0.2, 0.2))
    rates, par = ctx.abc_smc_propose(seed, idx0, n, prev, cum, sigma, **box)
    u = proposal_uniforms(seed, np.arange(n, dtype=np.uint64) + np.uint64(idx0))
    np.testing.assert_array_equal(par, np.searchsorted(cum, u[:, 0] * cum[-1], side="right"))
    np.testing.assert_array_equal(rates[:, 3], prev[par, 3])
    for k in range(2):  # the truncated normal drawn from the numpy uniforms, by scipy's inverse CDF
        lo, hi = RANGES[k]
        ref = np.array([_truncnorm(lo, hi, prev[j, k + 1], sigma[k]).ppf(uu) for j, uu in zip(par, u[:, k + 1])])
        err = np.abs(rates[:, k + 1].astype(np.float64) - ref)
        assert np.all(err <= 1e-5 * sigma[k] + np.spacing(np.float32(ref)).astype(np.float64)), float(err.max())
    for a in (1, 99, 100, 731):  # a block of draws gives the bits of the same indices in a longer block
        r2, p2 = ctx.abc_smc_propose(seed, idx0 + a, n - a, prev, cum, sigma, **box)
        np.testing.assert_array_equal(r2.view(np.uint32), rates[a:].view(np.uint32))
        np.testing.assert_array_equal(p2, par[a:])


# ---------------------------------------------------------------------------------------------------------------
# 3. the importance-sampling identity on the prior box
# ---------------------------------------------------------------------------------------------------------------
def _z(prev, sigma, ranges):
    z = np.ones(len(prev))
    for k, (lo, hi) in enumerate(ranges):
        if lo < hi and sigma[k] > 0:
            c = prev[:, k + 1].astype(np.float64)
            z *= special.ndtr((hi - c) / sigma[k]) - special.ndtr((lo - c) / sigma[k])
    return z


def _uniform_checks(theta, w):
    """Weighted estimates of expectations whose value under Uniform(box) is known: (name, estimate, truth, se).
    se is the larger of sqrt(var / ESS) and the delta-method sqrt(sum w^2 (f - estimate)^2)."""
    ess = 1.0 / np.sum(w * w)
    out = []

    def add(name, f, truth, var):
        est = float(np.dot(w, f))
        se = max(math.sqrt(var / ess), math.sqrt(float(np.dot(w * w, (f - est) ** 2))))
        out.append((name, est, truth, se))
    for k, (lo, hi) in enumerate(RANGES):
        x = theta[:, k]
        m2 = (lo * lo + lo * hi + hi * hi) / 3
        m4 = (hi ** 5 - lo ** 5) / (5 * (hi - lo))
        add(f"mean{k}", x, (lo + hi) / 2, (hi - lo) ** 2 / 12)
        add(f"m2_{k}", x * x, m2, m4 - m2 * m2)
        for q in (0.01, 0.05, 0.5, 0.95, 0.99):
            add(f"cdf{k}@{q}", (x < lo + q * (hi - lo)).astype(np.float64), q, q * (1 - q))
    c = 0.02 * 0.02
    add("corner", ((theta[:, 1] < 0.02 * 0.5) & (theta[:, 2] < 0.02 * 0.5)).astype(np.float64), c, c * (1 - c))
    return out, ess


@pytest.mark.gpu
@pytest.mark.parametrize("width", ["driver", "narrow"])
def test_importance_weights_represent_the_prior(ctx, width):
    rng = np.random.default_rng(7)
    M, N = 2000, 2_000_000
    prev = _edge_population(rng, M)
    W = rng.uniform(0.05, 1.0, M) ** 2
    W[: M // 3] *= 3.0
    W /= W.sum()
    th = prev[:, 1:].astype(np.float64)
    mean = W @ th
    sigma = np.sqrt(2.0 * (W @ (th - mean) ** 2))  # as the driver computes it
    if width == "narrow":
        sigma = sigma / 3
    sigma = tuple(float(s) for s in sigma)
    new, _ = ctx.abc_smc_propose(11, 5_000_000, N, prev, np.cumsum(W), sigma, **BOX)
    theta = new[:, 1:].astype(np.float64)
    w = ctx.abc_smc_weights(new, prev, W, sigma, **BOX)
    checks, ess = _uniform_checks(theta, w)
    z_with = max(abs(e - t) / s for _, e, t, s in checks)
    for name, est, truth, se in checks:
        assert abs(est - truth) <= 5 * se, (name, est, truth, se, ess)
    # power: weights W_j Z_j make the kernel's W_j / Z_j the plain W_j, the weights without the truncation correction
    wz = W * _z(prev, sigma, RANGES)
    w_noz = ctx.abc_smc_weights(new, prev, wz / wz.sum(), sigma, **BOX)
    bad, ess_noz = _uniform_checks(theta, w_noz)
    z_bad = {name: abs(e - t) / s for name, e, t, s in bad}
    print(f"{width}: sigma {sigma}, ESS {ess:.0f} of {N}; largest |z| with Z {z_with:.2f}; without Z: corner "
          f"{z_bad['corner']:.1f}, d0 cdf@0.01 {z_bad['cdf1@0.01']:.1f}, d1 cdf@0.01 {z_bad['cdf2@0.01']:.1f}, "
          f"b1 cdf@0.01 {z_bad['cdf0@0.01']:.1f} (ESS {ess_noz:.0f})")
    # Without Z the edges are over-weighted.  With the driver's width the kernels are wide, Z_j varies less over the
    # population and the bias is smaller; the narrow width shows it at the corner too.
    edges = {k: v for k, v in z_bad.items() if k.endswith("@0.01") or k == "corner"}
    assert max(edges.values()) > 5, edges  # the identity test fails without Z ...
    if width == "narrow":  # ... by a wide margin where the kernels are narrow
        assert z_bad["corner"] > 5 and min(z_bad[f"cdf{k}@0.01"] for k in range(3)) > 10, edges


# ---------------------------------------------------------------------------------------------------------------
# 4. the weight kernel against float64 within a bound derived from its arithmetic
# ---------------------------------------------------------------------------------------------------------------
# Per term W_j/Z_j * 2^-q_ij of S_i (abc_smc.cu smc_pair_kernel):
#  - f32(W_j / Z_j): relative u;
#  - q: d_k = (x_k - t_k) * sc_k from one f32 subtraction, one product and sc_k rounded to f32 (3u), squared in a
#    product or inside an FMA (one more u for d_1), summed by two FMAs (2u): |dq| <= 9u q (to first order; EX_Q adds
#    the second), which changes 2^-q by a factor exp(ln 2 |dq|);
#  - ex2.approx.ftz.f32: PTX ISA, "Floating Point Instructions: ex2": the maximum error is 2 ulp from the correctly
#    rounded result over the full range, so 2.5 ulp = 2.5 * 2^-23 relative to the exact power; a result below
#    2^-126 is flushed to 0, so a term with q near or above 126 may be lost entirely (counted at its full value);
#  - the tile sum: four partial sums of 32 FMAs, then two additions: gamma_34 of the terms (all >= 0);
#  - tiles added in f64, 1/S_i and the normalisation on the host in f64: (M / 128 + N + 2) * 2^-53, and the f64
#    reference itself (exp, the sums over M and N): another (8 q + 2 M + 2 N) * 2^-53.
EX2_REL = 2.5 * 2.0 ** -23
EX_Q = 9.0 * U32 * (1 + 1e-5)
GAMMA34 = 34 * U32 / (1 - 34 * U32)


def _free(sigma, ranges):
    return [k for k in range(3) if ranges[k][0] < ranges[k][1] and sigma[k] > 0]


def raw_sums_and_bounds(new, prev, w, sigma, ranges):
    """f64 S_i = sum_j (W_j / Z_j) exp(-sum_k (d_k / sigma_k)^2 / 2) over the free parameters, the bound B_i on
    |S_kernel_i - S_i| and the largest q = log2 of a term's factor that any term of S_i has."""
    free = _free(sigma, ranges)
    s = np.array([sigma[k] for k in free])
    p = prev[:, [k + 1 for k in free]].astype(np.float64)
    x = new[:, [k + 1 for k in free]].astype(np.float64)
    T = np.asarray(w, dtype=np.float64) / _z(prev, sigma, ranges)
    N, M = len(new), len(prev)
    S, B, qmax = np.zeros(N), np.zeros(N), np.zeros(N)
    step = max(1, 4_000_000 // M)
    for b in range(0, N, step):
        if free:
            q = (((x[b:b + step, None, :] - p[None, :, :]) / s) ** 2).sum(axis=2) / (2 * math.log(2))
        else:
            q = np.zeros((min(step, N - b), M))
        term = T[None, :] * np.exp2(-q)
        rel = (1 + U32) * (1 + EX2_REL) * np.exp(math.log(2) * EX_Q * q) * (1 + GAMMA34) - 1
        lost = q > 125.9
        S[b:b + step] = term.sum(axis=1)
        B[b:b + step] = (term * rel).sum(axis=1) + np.where(lost, term, 0.0).sum(axis=1)
        qmax[b:b + step] = q.max(axis=1)
    return S, B, qmax


def check_weights(got, new, prev, w, sigma, ranges):
    """Every normalised weight within the propagated bound; returns the largest observed / bound ratio."""
    S, B, qmax = raw_sums_and_bounds(new, prev, w, sigma, ranges)
    N, M = len(new), len(prev)
    r = B / S
    assert np.all(r < 0.5), r.max()
    rbar = r / (1 - r)  # |1/S_kernel - 1/S| <= rbar / S
    inv = 1.0 / S
    ref = inv / inv.sum()
    R = float(np.dot(rbar, inv) / inv.sum())  # the normaliser's relative error
    slack = (M / 128 + 3 * N + 2 * M + 8 * qmax + 16) * U64
    bound = (1 + rbar) / (1 - R) - 1 + slack
    err = np.abs(got / ref - 1)
    worst = float(np.max(err / bound))
    assert np.all(err <= bound), (int(np.argmax(err / bound)), worst)
    return worst


def _particles(rng, n):
    x = np.column_stack([np.ones(n), rng.uniform(1, 2, n), rng.uniform(0, 0.5, (n, 2))]).astype(np.float32)
    x[::5, 2] = 0.0
    x[1::5, 3] = 0.5
    x[2::5, 1] = 1.0 + rng.uniform(0, 0.01, len(x[2::5]))
    return x


SIGMA4 = (0.3, 0.1, 0.12)


@pytest.fixture(scope="module")
def worst_ratio():
    seen = []
    yield seen
    if seen:
        print(f"\nweight kernel: largest observed/bound ratio {max(seen):.3g} over {len(seen)} checks")


@pytest.mark.gpu
@pytest.mark.parametrize("N, M", [(1, 1), (1, 129), (127, 1), (128, 128), (129, 127), (300, 1000), (5000, 4097),
                                  (2000, 100_000)])
def test_weights_against_float64_at_tile_edges(ctx, worst_ratio, N, M):
    rng = np.random.default_rng(N * 7 + M)
    new, prev = _particles(rng, N), _particles(rng, M)
    w = rng.uniform(0.05, 1.0, M)
    w /= w.sum()
    got = ctx.abc_smc_weights(new, prev, w, SIGMA4, **BOX)
    assert got.shape == (N,) and np.all(np.isfinite(got)) and np.all(got > 0)
    worst_ratio.append(check_weights(got, new, prev, w, SIGMA4, RANGES))
    print(f"N {N} M {M}: observed/bound {worst_ratio[-1]:.3g}")


@pytest.mark.gpu
@pytest.mark.parametrize("mask", range(8))
def test_weights_fixed_parameters(ctx, worst_ratio, mask):
    """Bit k of mask: parameter k is free.  A fixed one is fixed by lo == hi (values on it) or by sigma = 0 (values
    anywhere in the range): it has no factor, whatever the values."""
    rng = np.random.default_rng(40 + mask)
    N, M = 300, 257
    new, prev = _particles(rng, N), _particles(rng, M)
    ranges, sigma = [list(r) for r in RANGES], list(SIGMA4)
    for k in range(3):
        if not mask >> k & 1:
            if k % 2 == 0:
                ranges[k] = [0.25 + k, 0.25 + k]
                new[:, k + 1] = prev[:, k + 1] = np.float32(0.25 + k)
            else:
                sigma[k] = 0.0
    w = rng.uniform(0.05, 1.0, M)
    w /= w.sum()
    box = dict(b1_range=tuple(ranges[0]), d0_range=tuple(ranges[1]), d1_range=tuple(ranges[2]))
    got = ctx.abc_smc_weights(new, prev, w, sigma, **box)
    assert len(_free(sigma, ranges)) == bin(mask).count("1")
    worst_ratio.append(check_weights(got, new, prev, w, sigma, ranges))
    if mask == 0:
        np.testing.assert_array_equal(got, np.full(N, got[0]))  # no factor at all: every S_i is sum_j W_j


@pytest.mark.gpu
def test_weights_do_not_depend_on_position(ctx):
    rng = np.random.default_rng(12)
    N, M = 1000, 300
    new, prev = _particles(rng, N), _particles(rng, M)
    w = rng.uniform(0.05, 1.0, M)
    w /= w.sum()
    base = ctx.abc_smc_weights(new, prev, w, SIGMA4, **BOX)
    tol = 8 * U64
    perm = rng.permutation(N)
    got = ctx.abc_smc_weights(new[perm], prev, w, SIGMA4, **BOX)
    first = int(np.nonzero(perm == 0)[0][0])
    np.testing.assert_allclose(got / got[first], base[perm] / base[0], rtol=tol, atol=0)
    sub = np.sort(np.concatenate([[0], rng.choice(np.arange(1, N), 136, replace=False)]))
    got = ctx.abc_smc_weights(new[sub], prev, w, SIGMA4, **BOX)
    np.testing.assert_allclose(got / got[0], base[sub] / base[0], rtol=tol, atol=0)
    got = ctx.abc_smc_weights(new[::-1][:777], prev, w, SIGMA4, **BOX)  # other blocks, other lanes
    np.testing.assert_allclose(got / got[0], base[::-1][:777] / base[N - 1], rtol=tol, atol=0)


@pytest.mark.gpu
def test_weights_fail_loudly(pkg, ctx, worst_ratio):
    prev = np.array([[1.0, 1.0, 0.0, 0.0], [1.0, 1.02, 0.01, 0.0]], dtype=np.float32)
    w = np.array([0.3, 0.7])
    sigma = (0.01, 0.01, 0.01)
    far = math.sqrt(2 * math.log(2))  # q = (d / sigma)^2 / (2 ln 2): q = 100 at d = sigma * 10 * far
    near = np.array([[1.0, 1.01, 0.005, 0.0]], dtype=np.float32)

    def at(q):  # a particle whose smallest q to the population is q (along b1, past the second parent)
        return np.array([[1.0, 1.02 + 0.01 * math.sqrt(q) * far, 0.01, 0.0]], dtype=np.float32)
    new = np.vstack([near, at(100.0)])
    got = ctx.abc_smc_weights(new, prev, w, sigma, **BOX)
    q = ((new[1, 1:].astype(np.float64) - prev[:, 1:]) / sigma) ** 2 / (2 * math.log(2))
    assert 99.9 < q.sum(axis=1).min() < 100.1 and got[1] > 0.999
    worst_ratio.append(check_weights(got, new, prev, w, sigma, RANGES))
    bad = {"q > 126 to every previous particle": (np.vstack([near, at(130.0)]), prev, w),
           "a NaN rate": (np.vstack([near, [[1.0, np.nan, 0.1, 0.1]]]).astype(np.float32), prev, w),
           "a NaN previous rate": (near, np.vstack([prev, [[1.0, 1.5, np.nan, 0.1]]]).astype(np.float32),
                                   np.array([0.3, 0.3, 0.4])),
           "all previous weights 0": (new, prev, np.zeros(2))}
    for what, (n_, p_, w_) in bad.items():
        with pytest.raises(pkg.EcdnaB200Error, match="status 1"):
            ctx.abc_smc_weights(n_, p_, w_, sigma, **BOX)
            pytest.fail(what)


# ---------------------------------------------------------------------------------------------------------------
# 5. a replay of the driver
# ---------------------------------------------------------------------------------------------------------------
WANT = ("stop_reason", "nminus", "nplus", "abc_distance", "abc_accept")


def replay_abc_smc(ctx, o, target, thresholds, M, quantile=0.5, max_generations=10, max_simulations=10_000_000,
                   b1_range=(1.0, 2.0), d0_range=(0.0, 0.5), d1_range=(0.0, 0.5), chunk=0, n_gpus=1):
    """DESIGN.md section 9 on the library's GPU primitives only; every host step in Python, sums sequential in index
    order in f64 (the host code is built without FMA contraction), the f32 steps in f32.  Returns the result dict of
    MultiContext.abc_smc plus "parent_pos": the parent of every particle as an index into the previous population."""
    thr = np.asarray(thresholds, dtype=np.float32)
    ranges = [b1_range, d0_range, d1_range]
    limit = max_simulations if max_simulations else UINT64_MAX
    eps, nxt, used, prev_rate = np.float32(np.inf), o.idx_begin, 0, 0.0
    sigma, cum, prev = [0.0, 0.0, 0.0], None, None
    gens, status = [], "max_generations"
    for g in range(max_generations):
        thr_g = [float(t * eps) if t > 0 else float(t) for t in thr]  # (f32 products)
        start = pos = nxt
        simulated, end, last_n = 0, 0, 0
        cur = {k: [] for k in ("idx", "parent_idx", "parent_pos", "rates", "distance", "cells", "rho")}
        while len(cur["idx"]) < M:
            acc = len(cur["idx"])
            left = limit - used - (pos - start)
            if left == 0:
                break
            n = chunk
            if n == 0:
                lo_n, hi_n = 4096 * n_gpus, 4 << 20
                rate = acc / simulated if simulated else prev_rate * quantile
                if rate > 0.0:
                    n = int(min(1.2 * (M - acc) / rate + 1.0, float(hi_n)))
                else:
                    n = 4 * last_n if last_n else lo_n
                n = min(max(n, lo_n), hi_n)
            n = min(n, left, 0xFFFFFFF0 - 1)
            last_n = n
            if g == 0:
                rates, parent = ctx.abc_draw_priors(o.seed, pos, n, o.b0, *ranges), None
            else:
                rates, parent = ctx.abc_smc_propose(o.seed, pos, n, prev["rates"], cum, sigma, *ranges)
            res = ctx.run(o, n_runs=n, idx_begin=pos, want=WANT, rates_per_run=rates,
                          abc_target=np.ascontiguousarray(target, dtype=np.uint64), abc_thresholds=thr_g,
                          snapshots=False)
            simulated += n
            rho = _rho(res.abc_distance, res.stop_reason, thr)
            ok = np.nonzero((res.abc_accept != 0) & np.isfinite(rho))[0][:M - acc]
            for i in ok:
                cur["idx"].append(pos + int(i))
                cur["parent_pos"].append(-1 if g == 0 else int(parent[i]))
                cur["parent_idx"].append(UINT64_MAX if g == 0 else prev["idx"][parent[i]])
                cur["rates"].append(rates[i])
                cur["distance"].append(res.abc_distance[i])
                cur["cells"].append(int(res.nminus[i]) + int(res.nplus[i]))
                cur["rho"].append(rho[i])
            if len(cur["idx"]) == M:
                end = pos + int(ok[-1]) + 1
            pos += n
        if len(cur["idx"]) < M:
            status = "budget"
            break
        consumed = end - start
        used += consumed
        nxt = end
        prev_rate = M / consumed
        cur["rates"] = np.array(cur["rates"], dtype=np.float32)
        cur["idx"] = np.array(cur["idx"], dtype=np.uint64)
        if g == 0:
            wts = np.full(M, 1.0 / M)
        else:
            wts = ctx.abc_smc_weights(cur["rates"], prev["rates"], prev["w"], sigma, *ranges)
        cur["w"] = wts
        w2 = 0.0
        for x in wts.tolist():
            w2 += x * x
        gens.append(dict(cur, epsilon=eps, consumed=consumed, simulated=simulated, ess=1.0 / w2))
        if eps == np.float32(1.0):
            status = "reached"
            break
        wl = wts.tolist()
        for k in range(3):
            th = cur["rates"][:, k + 1].astype(np.float64).tolist()
            mean = 0.0
            for a, b in zip(wl, th):
                mean += a * b
            var = 0.0
            for a, b in zip(wl, th):
                d = b - mean
                var += a * d * d
            sigma[k] = math.sqrt(2.0 * var)
        c, cum = 0.0, np.zeros(M)
        for i, a in enumerate(wl):
            c += a
            cum[i] = c
        kq = min(M, max(1, int(math.ceil(quantile * M))))
        rho_k = np.sort(np.array(cur["rho"], dtype=np.float32))[kq - 1]
        eps = np.float32(min(eps, max(np.float32(1.0), rho_k)))
        prev = cur
    G = len(gens)
    out = {"generations": G, "status": status,
           "idx": np.array([x["idx"] for x in gens], dtype=np.uint64).reshape(G, M),
           "parent_idx": np.array([x["parent_idx"] for x in gens], dtype=np.uint64).reshape(G, M),
           "parent_pos": np.array([x["parent_pos"] for x in gens], dtype=np.int64).reshape(G, M),
           "rates": np.array([x["rates"] for x in gens], dtype=np.float32).reshape(G, M, 4),
           "distance": np.array([x["distance"] for x in gens], dtype=np.float32).reshape(G, M, 4),
           "weight": np.array([x["w"] for x in gens], dtype=np.float64).reshape(G, M),
           "cells": np.array([x["cells"] for x in gens], dtype=np.uint64).reshape(G, M)}
    for k, dt in (("epsilon", np.float32), ("consumed", np.uint64), ("simulated", np.uint64), ("ess", np.float64)):
        out[k] = np.array([x[k] for x in gens], dtype=dt)
    return out


@pytest.fixture(scope="module")
def problem(pkg):
    o = pkg.SimulationOptions(b0=1.0, b1=1.4, d0=0.2, d1=0.2, cells=2000, runs=1, save_snapshots=False)
    return o, ob.run(oracle_opts(o, 260), hist_cap=BINS).hist


@pytest.fixture(scope="module")
def mc(pkg):
    m = pkg.MultiContext([0])
    yield m
    m.close()


TIGHT = (0.05, 0.1, 0.1, 0.1)  # (C4's thresholds: eps stays above 1 for a few generations)
REPLAY = {
    "auto-chunk": dict(thresholds=TIGHT, max_generations=4),
    "chunk-333": dict(thresholds=TIGHT, max_generations=4, chunk=333, quantile=0.333),  # (k = ceil(66.6) = 67)
    "disabled-threshold": dict(thresholds=(0.05, -1.0, 0.1, 0.1), max_generations=4, quantile=0.7),
    "zero-threshold": dict(thresholds=(0.05, 0.1, 0.1, 0.0), max_generations=3, max_simulations=9000),
    "fixed-d1": dict(thresholds=TIGHT, max_generations=4, chunk=2000, d1_range=(0.2, 0.2)),
}


def _compare(r, ref):
    assert r["generations"] == ref["generations"] and r["status"] == ref["status"], (r["status"], ref["status"])
    for k in ("idx", "parent_idx", "rates", "distance", "weight", "cells", "epsilon", "consumed", "simulated", "ess"):
        x, y = np.ascontiguousarray(r[k]), np.ascontiguousarray(ref[k])
        assert x.shape == y.shape, (k, x.shape, y.shape)
        np.testing.assert_array_equal(x.view(np.uint8), y.view(np.uint8), err_msg=k)
    for t in range(1, ref["generations"]):  # the reported parent is the one the proposal drew
        np.testing.assert_array_equal(r["parent_idx"][t], ref["idx"][t - 1][ref["parent_pos"][t]])


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(REPLAY))
def test_driver_matches_replay(ctx, mc, problem, case):
    o, target = problem
    kw = dict(REPLAY[case])
    thr = kw.pop("thresholds")
    r = mc.abc_smc(o, target, thr, 200, **kw)
    ref = replay_abc_smc(ctx, o, target, thr, 200, **kw)
    _compare(r, ref)
    if case == "zero-threshold":  # no distance of this problem is ever exactly 0: the budget ends generation 0
        assert r["status"] == "budget" and r["generations"] == 0
    else:
        assert r["generations"] >= 3, r["epsilon"]
    if "d1_range" in kw:
        assert np.all(r["rates"][:, :, 3] == np.float32(0.2))
    print(f"{case}: eps {r['epsilon'].tolist()} consumed {r['consumed'].tolist()} simulated {r['simulated'].tolist()}")


@pytest.mark.gpu
def test_driver_matches_replay_when_the_budget_ends_generation_2(ctx, mc, problem):
    o, target = problem
    full = mc.abc_smc(o, target, TIGHT, 200, max_generations=4)
    assert full["generations"] >= 3
    budget = int(full["consumed"][:2].sum()) + int(full["consumed"][2]) // 2
    r = mc.abc_smc(o, target, TIGHT, 200, max_generations=4, max_simulations=budget)
    ref = replay_abc_smc(ctx, o, target, TIGHT, 200, max_generations=4, max_simulations=budget)
    _compare(r, ref)
    assert r["status"] == "budget" and r["generations"] == 2
