"""The correlated ABC-SMC kernels on the GPU (ecdna_b200_abc_smc_propose_cov / _weights_cov / ecdna_b200_abc_smc_ex,
DESIGN.md section 9) against the numpy and mpmath restatement of test_abc_smc_kernels_host.py: a diagonal Sigma is the
component kernel bit for bit, every proposal maps back to its own Philox uniforms through the exact Rosenblatt
transform (far tails included), the weighted proposals represent the prior, the weights agree with float64 within a
bound derived from the kernel's arithmetic, a Python replay of the driver matches it byte for byte, the posterior at
eps = 1 matches rejection ABC, and the CLI writes what write_abc_smc writes."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest
from scipy import stats

import oracle_binding as ob
from test_abc_smc_kernels_host import TRI, free_params, kernel_log_density, log_mass, olcm_closed_form, pack, rosenblatt
from test_gpu_abc_smc import BINS, BOX, THR, UINT64_MAX, _rejection, _rho
from test_gpu_abc_smc_reference import _edge_population, _uniform_checks, proposal_uniforms
from test_gpu_parity import oracle_opts

pytestmark = pytest.mark.gpu
RANGES = [BOX["b1_range"], BOX["d0_range"], BOX["d1_range"]]
U32 = 2.0 ** -24
U64 = 2.0 ** -53
LOG2PI = math.log2(2 * math.pi)


def _cov(sd, r12=0.0, r13=0.0, r23=0.0):
    R = np.array([[1, r12, r13], [r12, 1, r23], [r13, r23, 1]], dtype=np.float64)
    return pack(np.outer(sd, sd) * R)


def _box(ranges):
    return dict(b1_range=tuple(ranges[0]), d0_range=tuple(ranges[1]), d1_range=tuple(ranges[2]))


# ---------------------------------------------------------------------------------------------------------------
# 1. a diagonal Sigma is the component kernel
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("sd", [(0.3, 0.1, 0.12), (0.02, 0.004, 0.01), (2.0, 1.5, 3.0)])
def test_diagonal_sigma_is_the_component_kernel(ctx, sd):
    rng = np.random.default_rng(1)
    M, n = 300, 100_000
    prev = _edge_population(rng, M)  # (a third of the parents on or near d0 = 0)
    W = rng.uniform(0.1, 1, M)
    W /= W.sum()
    cum = np.cumsum(W)
    cov = pack(np.diag(np.square(sd)))
    sigma = tuple(float(x) for x in np.sqrt(cov[[TRI[(k, k)] for k in range(3)]]))
    for box in (BOX, dict(BOX, d1_range=(0.2, 0.2))):
        want_r, want_p = ctx.abc_smc_propose(3, 2**32 - 77, n, prev, cum, sigma, **box)
        for c in (cov, np.tile(cov, (M, 1))):
            r, p = ctx.abc_smc_propose_cov(3, 2**32 - 77, n, prev, cum, c, **box)
            np.testing.assert_array_equal(p, want_p)
            np.testing.assert_array_equal(r.view(np.uint32), want_r.view(np.uint32))
    new = want_r[:2000]
    got = ctx.abc_smc_weights_cov(new, prev, W, cov, **BOX)
    check_weights(got, new, prev, W, cov, RANGES)
    comp = ctx.abc_smc_weights(new, prev, W, sigma, **BOX)
    np.testing.assert_allclose(got, comp, rtol=1e-4, atol=0)  # (two f32 paths, each within its own bound)


# ---------------------------------------------------------------------------------------------------------------
# 2-3. proposals against the exact kernel: Rosenblatt transform back to the Philox uniforms
# ---------------------------------------------------------------------------------------------------------------
def check_rosenblatt(rates, par, prev, cov, ranges, seed, idx0):
    """Every draw's Rosenblatt transform, computed from its rounded theta in f64, returns the uniforms of its Philox
    words.  Bound: theta_t is m_t + L_tt z rounded once to f32 (and clamped into the box), so e_t moves by at most
    ulp(theta_t) / (2 L_tt) and u_t by the truncated density there times that (x2 for its variation over one ulp),
    plus the f64 rounding of e and a (relative 1e-15 of their size, times the density) and 1e-9 for the f64 inverse
    CDF.  Returns the transformed uniforms."""
    n = len(rates)
    u = proposal_uniforms(seed, np.arange(n, dtype=np.uint64) + np.uint64(idx0))
    free = free_params(ranges, cov)
    assert np.all(np.isfinite(rates))
    for k in range(3):
        lo, hi = ranges[k]
        assert np.all((rates[:, k + 1] >= np.float32(lo)) & (rates[:, k + 1] <= np.float32(hi))), k
        if k not in free:
            np.testing.assert_array_equal(rates[:, k + 1], prev[par, k + 1])
    cov = np.asarray(cov, dtype=np.float64).reshape(-1, 6)
    out = np.zeros((n, len(free)))
    for j in np.unique(par):
        sel = par == j
        cj = cov[j] if len(cov) > 1 else cov[0]
        ur, e, a, b, L = rosenblatt(rates[sel, 1:], prev[j, 1:], cj, ranges)
        for t, k in enumerate(free):
            th = rates[sel, k + 1]
            dens = np.exp(-0.5 * e[:, t] ** 2 - log_mass(a[:, t], b[:, t])) / math.sqrt(2 * math.pi)
            bound = dens * (2 * np.spacing(th).astype(np.float64) / L[t, t] + 1e-15 * (np.abs(e[:, t]) + np.abs(a[:, t]))) + 1e-9
            err = np.abs(ur[:, t] - u[sel, k + 1])
            assert np.all(err <= bound), (j, k, float(np.max(err / bound)), float(np.max(err)))
        out[sel] = ur
    return out


SINGLE = {"interior": (1.5, 0.25, 0.2), "edge": (1.3, 0.0, 0.3), "corner": (1.0, 0.0, 0.0)}


@pytest.mark.parametrize("rho", [0.0, 0.9, -0.99, 0.999])
@pytest.mark.parametrize("where", sorted(SINGLE))
def test_proposals_against_the_exact_kernel(ctx, where, rho):
    prev = np.array([[1.0, *SINGLE[where]]], dtype=np.float32)
    cov = _cov((0.25, 0.12, 0.1), r12=0.03, r23=rho)
    n, seed, idx0 = 200_000, 17, 2**32 - 5000
    rates, par = ctx.abc_smc_propose_cov(seed, idx0, n, prev, np.array([1.0]), cov, **BOX)
    assert np.all(par == 0) and np.all(rates[:, 0] == 1.0)
    ur = check_rosenblatt(rates, par, prev, cov, RANGES, seed, idx0)
    for t in range(3):
        p = stats.kstest(ur[:, t], "uniform").pvalue
        assert p > 1e-3, (t, p)
    s, c = math.sqrt(cov[0]), float(prev[0, 1])
    p = stats.kstest(rates[:, 1].astype(np.float64), stats.truncnorm((1.0 - c) / s, (2.0 - c) / s, loc=c, scale=s).cdf).pvalue
    assert p > 1e-3, p


@pytest.mark.parametrize("K", [5.0, 37.0, 1e2, 1e4])
def test_far_tails(ctx, K):
    """A parent outside the box in d1 by K conditional sds (below lo and above hi), d0 correlated at 0.9 with it and
    b1 fixed: the conditional intervals of d1 lie K -+ 10 sds out."""
    ranges = [(1.5, 1.5), (0.0, 0.5), (0.0, 0.5)]
    cov = _cov((1.0, 0.05, 0.05), r23=0.9)
    L22 = 0.05 * math.sqrt(1 - 0.81)
    for side, c2 in (("below", 0.0 - K * L22), ("above", 0.5 + K * L22)):
        prev = np.array([[1.0, 1.5, 0.25, c2]], dtype=np.float32)
        n, seed = 100_000, 23
        rates, par = ctx.abc_smc_propose_cov(seed, 1000, n, prev, np.array([1.0]), cov, **_box(ranges))
        check_rosenblatt(rates, par, prev, cov, ranges, seed, 1000)


# ---------------------------------------------------------------------------------------------------------------
# 4. the importance-sampling identity on the prior box
# ---------------------------------------------------------------------------------------------------------------
def _spread_correlated_population(rng, M):
    """test_gpu_abc_smc_reference's population crowded against d0 = 0 and the (b1 = 1, d1 = 0) corner, a third spread
    over the box, with d1 pulled towards d0 and b1 tilted against d0."""
    x = _edge_population(rng, M)
    x[:, 3] = np.clip(0.5 * x[:, 3] + 0.5 * x[:, 2], 0, 0.5)
    x[:, 1] = np.clip(x[:, 1] + 0.8 * x[:, 2], 1, 2)
    return x


def _correlated_population(rng, M):
    """Against d0 = 0 and d1 = 0, d1 following d0: corr(d0, d1) ~ 0.95, b1 tilted against d0."""
    d0 = np.abs(rng.normal(0, 0.06, M))
    d1 = np.clip(0.9 * d0 + rng.normal(0, 0.015, M), 0, 0.5)
    b1 = np.clip(1.3 + 1.5 * d0 + rng.normal(0, 0.05, M), 1, 2)
    return np.column_stack([np.ones(M), b1, d0, d1]).astype(np.float32)


def _sigmas(kind, prev, W, rng):
    th = prev[:, 1:].astype(np.float64)
    if kind == "mvn":
        m = W @ th
        return 2.0 * pack((W[:, None] * (th - m)).T @ (th - m))
    sel = rng.uniform(size=len(W)) < 0.5
    return np.stack([pack(olcm_closed_form(th, W, sel, j)) for j in range(len(W))])


def _sums_without_masses(new, prev, W, cov):
    """sum_j W_j N(theta_i; c_j, Sigma_j) in f64 over all three parameters: the kernel's density without any
    truncation mass."""
    cov = np.asarray(cov, dtype=np.float64).reshape(-1, 6)
    Li = np.linalg.inv(np.linalg.cholesky(np.stack([olcm_unpack(c) for c in cov])))
    logdet = np.log(np.diagonal(np.linalg.cholesky(np.stack([olcm_unpack(c) for c in cov])), axis1=1, axis2=2)).sum(1)
    c = prev[:, 1:].astype(np.float64)
    x = new[:, 1:].astype(np.float64)
    S = np.zeros(len(x))
    for b in range(0, len(x), 10_000):
        d = x[b:b + 10_000, None, :] - c[None, :, :]
        e = np.einsum("mij,nmj->nmi", Li, d) if len(cov) > 1 else d @ Li[0].T
        S[b:b + 10_000] = (W * np.exp(-0.5 * (e * e).sum(axis=2) - logdet)).sum(axis=1)
    return S


@pytest.mark.parametrize("kind", ["mvn", "olcm"])
def test_importance_weights_represent_the_prior(ctx, kind):
    rng = np.random.default_rng(31)
    M, N = 300, 1_000_000
    prev = _spread_correlated_population(rng, M)
    W = rng.uniform(0.2, 1.0, M)
    W /= W.sum()
    cov = _sigmas(kind, prev, W, rng)
    new, _ = ctx.abc_smc_propose_cov(41, 7_000_000, N, prev, np.cumsum(W), cov, **BOX)
    w = ctx.abc_smc_weights_cov(new, prev, W, cov, **BOX)
    checks, ess = _uniform_checks(new[:, 1:].astype(np.float64), w)
    for name, est, truth, se in checks:
        assert abs(est - truth) <= 5 * se, (name, est, truth, se, ess)
    # power: the same identity with every truncation mass dropped (the weights in f64 numpy, first 300 000 draws)
    # fails: a CPU restatement of this check put it 25 SE off at 10^6 draws, ~14 at 300 000
    sub = new[:300_000]
    inv = 1.0 / _sums_without_masses(sub, prev, W, cov)
    bad, ess_bad = _uniform_checks(sub[:, 1:].astype(np.float64), inv / inv.sum())
    z = {name: abs(e - t) / s for name, e, t, s in bad}
    print(f"{kind}: ESS {ess:.0f} of {N}; largest |z| {max(abs(e - t) / s for _, e, t, s in checks):.2f}; "
          f"without the masses: largest |z| {max(z.values()):.1f} ({max(z, key=z.get)})")
    assert max(z.values()) > 5, z


# ---------------------------------------------------------------------------------------------------------------
# 5. the weights against float64 within a bound derived from the kernel's arithmetic
# ---------------------------------------------------------------------------------------------------------------
# smc_pair_cov_kernel computes the log2 of each term in f64 (whitening, the truncated factors in the factored form,
# log2 W_j - sum log2 L_tt - log2 of the first mass from the tiles kernel), relative to shift = max_j of that log2
# weight: x_ij = log2(W_j q_j(theta_i)) + D log2(2 pi) / 2 - shift.  Per term:
#  - the f64 evaluation: at most 1e-12 (1 + |x|) in x (a few dozen operations on magnitudes <= |x| + 40, each
#    2^-53 relative, with erfcx, log, normcdf within a few ulp);
#  - x rounded to f32: |dx| <= 2^-24 |x|; both change 2^x by a factor exp(ln 2 |dx|);
#  - ex2.approx.ftz.f32: 2 ulp from the correctly rounded result (PTX ISA), 2.5 * 2^-23 relative; below 2^-126 the
#    result is flushed to 0 (such a term counts at its full value);
#  - the tile sum: four partial sums of 32 additions, then two: gamma_34 of the terms (all >= 0);
#  - the tiles added in f64, 1/S_i and the normalisation on the host: as in test_gpu_abc_smc_reference.py.
EX2_REL = 2.5 * 2.0 ** -23
GAMMA34 = 34 * U32 / (1 - 34 * U32)


def raw_sums_and_bounds(new, prev, W, cov, ranges):
    cov = np.asarray(cov, dtype=np.float64).reshape(-1, 6)
    free = free_params(ranges, cov)
    D = len(free)
    lt = np.zeros((len(new), len(prev)))  # log2(W_j q_j(theta_i)) + D log2(2 pi) / 2
    logw = np.zeros(len(prev))
    for j in range(len(prev)):
        cj = cov[j] if len(cov) > 1 else cov[0]
        with np.errstate(divide="ignore"):
            lt[:, j] = (kernel_log_density(new[:, 1:], prev[j, 1:], cj, ranges) / math.log(2) + math.log2(W[j])
                        + D * LOG2PI / 2)
        if D:
            Lj = np.linalg.cholesky(np.asarray(olcm_unpack(cj))[np.ix_(free, free)])
            lo, hi = ranges[free[0]]
            c0 = float(prev[j, free[0] + 1])
            lm = float(log_mass((lo - c0) / Lj[0, 0], (hi - c0) / Lj[0, 0]))
            logw[j] = math.log2(W[j]) - float(np.sum(np.log2(np.diag(Lj)))) - lm / math.log(2)
        else:
            logw[j] = math.log2(W[j])
    shift = logw.max()
    x = lt - shift
    term = np.exp2(x)
    dx = 1e-12 * (1 + np.abs(x)) + U32 * np.abs(x)
    rel = np.exp(math.log(2) * dx) * (1 + EX2_REL) * (1 + GAMMA34) - 1
    lost = x < -125.9
    return term.sum(axis=1), (term * rel).sum(axis=1) + np.where(lost, term, 0.0).sum(axis=1)


def olcm_unpack(c):
    S = np.zeros((3, 3))
    for (r, q), i in TRI.items():
        S[r, q] = S[q, r] = c[i]
    return S


def check_weights(got, new, prev, W, cov, ranges):
    S, B = raw_sums_and_bounds(new, prev, W, cov, ranges)
    N, M = len(new), len(prev)
    r = B / S
    assert np.all(r < 0.5), r.max()
    rbar = r / (1 - r)
    inv = 1.0 / S
    ref = inv / inv.sum()
    R = float(np.dot(rbar, inv) / inv.sum())
    slack = (M / 128 + 3 * N + 2 * M + 64) * U64
    bound = (1 + rbar) / (1 - R) - 1 + slack
    err = np.abs(got / ref - 1)
    worst = float(np.max(err / bound))
    assert np.all(err <= bound), (int(np.argmax(err / bound)), worst)
    return worst


def _particles(rng, n):
    x = _correlated_population(rng, n)
    x[::7, 2] = 0.0
    x[1::7, 3] = 0.5
    return x


@pytest.mark.parametrize("N, M, per_parent", [(1, 1, False), (129, 1, True), (300, 129, False), (300, 129, True),
                                              (1000, 300, True), (257, 1000, False)])
def test_weights_against_float64(ctx, N, M, per_parent):
    rng = np.random.default_rng(N + 3 * M)
    new, prev = _particles(rng, N), _particles(rng, M)
    W = rng.uniform(0.05, 1.0, M)
    W /= W.sum()
    cov = _sigmas("olcm", prev, W, rng) if per_parent else _sigmas("mvn", prev, W, rng)
    if M == 1:  # (one particle has no covariance)
        cov = _cov((0.3, 0.1, 0.08), -0.5, 0.2, 0.6)
        cov = np.tile(cov, (1, 1)) if per_parent else cov
    got = ctx.abc_smc_weights_cov(new, prev, W, cov, **BOX)
    assert got.shape == (N,) and np.all(got > 0)
    print(f"N {N} M {M} per-parent {per_parent}: observed/bound {check_weights(got, new, prev, W, cov, RANGES):.3g}")


@pytest.mark.parametrize("mask", range(8))
def test_weights_free_fixed_masks(ctx, mask):
    """Bit k of mask: parameter k is free.  A fixed one is fixed by lo == hi (k = 0, 2) or by variance 0 (k = 1)."""
    rng = np.random.default_rng(60 + mask)
    N, M = 200, 150
    new, prev = _particles(rng, N), _particles(rng, M)
    W = rng.uniform(0.05, 1.0, M)
    W /= W.sum()
    ranges = [list(r) for r in RANGES]
    cov = olcm_unpack(_cov((0.3, 0.1, 0.08), -0.5, 0.2, 0.6))
    for k in range(3):
        if not mask >> k & 1:
            if k != 1:
                ranges[k] = [0.25 + k, 0.25 + k]
                new[:, k + 1] = prev[:, k + 1] = np.float32(0.25 + k)
                cov[k, :] = cov[:, k] = np.nan  # (ignored)
            else:
                cov[k, :] = cov[:, k] = 0.0
    cov = pack(cov)
    assert len(free_params(ranges, cov)) == bin(mask).count("1")
    for c in (cov, np.tile(cov, (M, 1))):
        got = ctx.abc_smc_weights_cov(new, prev, W, c, **_box(ranges))
        check_weights(got, new, prev, W, np.nan_to_num(c), ranges)
        if mask == 0:
            np.testing.assert_array_equal(got, np.full(N, got[0]))


def test_weights_do_not_depend_on_position(ctx):
    rng = np.random.default_rng(12)
    N, M = 1000, 300
    new, prev = _particles(rng, N), _particles(rng, M)
    W = rng.uniform(0.05, 1.0, M)
    W /= W.sum()
    cov = _sigmas("olcm", prev, W, rng)
    base = ctx.abc_smc_weights_cov(new, prev, W, cov, **BOX)
    perm = rng.permutation(N)
    got = ctx.abc_smc_weights_cov(new[perm], prev, W, cov, **BOX)
    first = int(np.nonzero(perm == 0)[0][0])
    np.testing.assert_allclose(got / got[first], base[perm] / base[0], rtol=8 * U64, atol=0)
    got = ctx.abc_smc_weights_cov(new[::-1][:777], prev, W, cov, **BOX)
    np.testing.assert_allclose(got / got[0], base[::-1][:777] / base[N - 1], rtol=8 * U64, atol=0)
    again = ctx.abc_smc_weights_cov(new, prev, W, cov, **BOX)
    np.testing.assert_array_equal(again.view(np.uint64), base.view(np.uint64))


def test_bad_sigma_is_an_error(pkg, ctx):
    rng = np.random.default_rng(13)
    prev = _particles(rng, 10)
    W = np.full(10, 0.1)
    good = _cov((0.3, 0.1, 0.08), -0.5, 0.2, 0.6)
    bad = {"not positive definite": _cov((0.3, 0.1, 0.08), 0.9, 0.9, -0.9),
           "a NaN entry": np.where(np.arange(6) == 4, np.nan, good),
           "n_cov = 2": np.tile(good, (2, 1)),
           "variance 0 in some Sigma only": np.vstack([good] * 9 + [np.where(np.arange(6) == 2, 0.0, good)]),
           "a negative variance": np.where(np.arange(6) == 0, -1.0, good)}
    for what, c in bad.items():
        with pytest.raises(pkg.EcdnaB200Error, match="status 1"):
            ctx.abc_smc_weights_cov(prev, prev, W, c, **BOX)
            pytest.fail(what)
        with pytest.raises(pkg.EcdnaB200Error, match="status 1"):
            ctx.abc_smc_propose_cov(1, 0, 10, prev, np.cumsum(W), c, **BOX)
            pytest.fail(what)


# ---------------------------------------------------------------------------------------------------------------
# 6. the driver
# ---------------------------------------------------------------------------------------------------------------
WANT = ("stop_reason", "nminus", "nplus", "abc_distance", "abc_accept")
KERNELS = ["component", "mvn", "olcm"]


def _usable(cov, ranges):
    """A Sigma the driver uses: valid for the _cov calls, every pivot L_tt >= 2^-12 (hi - lo)."""
    cov = np.asarray(cov).reshape(-1, 6)
    for k in range(3):
        if ranges[k][0] < ranges[k][1]:
            pos = cov[:, TRI[(k, k)]] > 0
            if pos.any() and not pos.all():
                return False
    free = free_params(ranges, cov)
    for c in cov:
        S = olcm_unpack(c)[np.ix_(free, free)]
        try:
            L = np.linalg.cholesky(S)
        except np.linalg.LinAlgError:
            return False
        if any(L[t, t] < 2.0 ** -12 * (ranges[k][1] - ranges[k][0]) for t, k in enumerate(free)):
            return False
    return True


def _seq_sum(xs):
    s = 0.0
    for x in xs:
        s += x
    return s


def replay(ctx, o, target, thresholds, M, kernel, quantile=0.5, max_generations=10, max_simulations=10_000_000,
           chunk=0, **box):
    """DESIGN.md section 9 with the correlated kernels, on the library's GPU primitives only: every host step in
    Python, sums sequential in index order in f64."""
    thr = np.asarray(thresholds, dtype=np.float32)
    ranges = [box.get("b1_range", (1.0, 2.0)), box.get("d0_range", (0.0, 0.5)), box.get("d1_range", (0.0, 0.5))]
    limit = max_simulations or UINT64_MAX
    eps, nxt, used, prev_rate = np.float32(np.inf), o.idx_begin, 0, 0.0
    sigma, cov, use, cum, prev = [0.0] * 3, None, "component", None, None
    gens, status = [], "max_generations"
    for g in range(max_generations):
        thr_g = [float(t * eps) if t > 0 else float(t) for t in thr]
        start = pos = nxt
        simulated, end, last_n = 0, 0, 0
        cur = {k: [] for k in ("idx", "parent_idx", "rates", "distance", "cells", "rho")}
        while len(cur["idx"]) < M:
            acc = len(cur["idx"])
            left = limit - used - (pos - start)
            if left == 0:
                break
            n = chunk
            if n == 0:
                lo_n, hi_n = 4096, 4 << 20
                rate = acc / simulated if simulated else prev_rate * quantile
                n = int(min(1.2 * (M - acc) / rate + 1.0, float(hi_n))) if rate > 0 else (4 * last_n if last_n else lo_n)
                n = min(max(n, lo_n), hi_n)
            n = min(n, left, 0xFFFFFFF0 - 1)
            last_n = n
            if g == 0:
                rates, parent = ctx.abc_draw_priors(o.seed, pos, n, o.b0, *ranges), None
            elif use == "component":
                rates, parent = ctx.abc_smc_propose(o.seed, pos, n, prev["rates"], cum, sigma, *ranges)
            else:
                rates, parent = ctx.abc_smc_propose_cov(o.seed, pos, n, prev["rates"], cum, cov, *ranges)
            res = ctx.run(o, n_runs=n, idx_begin=pos, want=WANT, rates_per_run=rates,
                          abc_target=np.ascontiguousarray(target, dtype=np.uint64), abc_thresholds=thr_g,
                          snapshots=False)
            simulated += n
            rho = _rho(res.abc_distance, res.stop_reason, thr)
            ok = np.nonzero((res.abc_accept != 0) & np.isfinite(rho))[0][:M - acc]
            for i in ok:
                cur["idx"].append(pos + int(i))
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
        elif use == "component":
            wts = ctx.abc_smc_weights(cur["rates"], prev["rates"], prev["w"], sigma, *ranges)
        else:
            wts = ctx.abc_smc_weights_cov(cur["rates"], prev["rates"], prev["w"], cov, *ranges)
        cur["w"] = wts
        gens.append(dict(cur, epsilon=eps, consumed=consumed, simulated=simulated,
                         ess=1.0 / _seq_sum([x * x for x in wts.tolist()]), used=None if g == 0 else use))
        if eps == np.float32(1.0):
            status = "reached"
            break
        wl = wts.tolist()
        th = [cur["rates"][:, k + 1].astype(np.float64).tolist() for k in range(3)]
        mean = [_seq_sum([a * b for a, b in zip(wl, th[k])]) for k in range(3)]
        S = np.zeros(6)
        for k in range(3):
            for l in range(k + 1):
                v = 0.0
                for i, a in enumerate(wl):
                    v += a * (th[k][i] - mean[k]) * (th[l][i] - mean[l])
                S[TRI[(k, l)]] = 2.0 * v
            sigma[k] = math.sqrt(S[TRI[(k, k)]])
        c, cum = 0.0, np.zeros(M)
        for i, a in enumerate(wl):
            c += a
            cum[i] = c
        kq = min(M, max(1, int(math.ceil(quantile * M))))
        eps = np.float32(min(eps, max(np.float32(1.0), np.sort(np.array(cur["rho"], dtype=np.float32))[kq - 1])))
        use = "component"
        if kernel == "olcm":
            sel = [i for i in range(M) if cur["rho"][i] <= eps]
            sw = _seq_sum([wl[i] for i in sel])
            m = [_seq_sum([wl[i] / sw * th[k][i] for i in sel]) for k in range(3)]
            Cm = np.zeros(6)
            for k in range(3):
                for l in range(k + 1):
                    Cm[TRI[(k, l)]] = _seq_sum([wl[i] / sw * (th[k][i] - m[k]) * (th[l][i] - m[l]) for i in sel])
            cov = np.zeros((M, 6))
            for j in range(M):
                for k in range(3):
                    for l in range(k + 1):
                        cov[j, TRI[(k, l)]] = Cm[TRI[(k, l)]] + (m[k] - th[k][j]) * (m[l] - th[l][j])
            if _usable(cov, ranges):
                use = "olcm"
        if kernel != "component" and use == "component":
            cov = S.copy()
            if _usable(cov, ranges):
                use = "mvn"
        prev = cur
    G = len(gens)
    out = {"generations": G, "status": status, "kernel_used": [x["used"] for x in gens]}
    for k, dt, shape in (("idx", np.uint64, (G, M)), ("parent_idx", np.uint64, (G, M)), ("rates", np.float32, (G, M, 4)),
                         ("distance", np.float32, (G, M, 4)), ("w", np.float64, (G, M)), ("cells", np.uint64, (G, M))):
        out["weight" if k == "w" else k] = np.array([x[k] for x in gens], dtype=dt).reshape(shape)
    for k, dt in (("epsilon", np.float32), ("consumed", np.uint64), ("simulated", np.uint64), ("ess", np.float64)):
        out[k] = np.array([x[k] for x in gens], dtype=dt)
    return out


def _same(r, ref, extra=("simulated",)):
    """Byte for byte (draws simulated past a generation's M-th acceptance depend on the chunk size: extra=())."""
    assert r["generations"] == ref["generations"] and r["status"] == ref["status"], (r["status"], ref["status"])
    assert r["kernel_used"] == ref["kernel_used"], (r["kernel_used"], ref["kernel_used"])
    for k in ("idx", "parent_idx", "rates", "distance", "weight", "cells", "epsilon", "consumed", "ess") + extra:
        x, y = np.ascontiguousarray(r[k]), np.ascontiguousarray(ref[k])
        assert x.shape == y.shape, (k, x.shape, y.shape)
        np.testing.assert_array_equal(x.view(np.uint8), y.view(np.uint8), err_msg=k)


@pytest.fixture(scope="module")
def problem(pkg):
    o = pkg.SimulationOptions(b0=1.0, b1=1.4, d0=0.2, d1=0.2, cells=2000, runs=1, save_snapshots=False)
    return o, ob.run(oracle_opts(o, 260), hist_cap=BINS).hist


@pytest.fixture(scope="module")
def mc(pkg):
    m = pkg.MultiContext([0])
    yield m
    m.close()


TIGHT = (0.05, 0.1, 0.1, 0.1)
REPLAY = {
    "mvn": ("mvn", TIGHT, dict(max_generations=4)),
    "mvn-fixed-d1": ("mvn", TIGHT, dict(max_generations=4, chunk=2000, d1_range=(0.2, 0.2))),
    "olcm": ("olcm", TIGHT, dict(max_generations=4)),
    "olcm-fixed-b1-chunk-333": ("olcm", TIGHT, dict(max_generations=4, chunk=333, quantile=0.333, b1_range=(1.4, 1.4))),
    # thresholds no particle meets and ceil(alpha M) = 1: one particle within eps, C = 0, Sigma_j of rank 1 -> mvn
    "olcm-forced-fallback": ("olcm", (0.0005, 0.001, 0.001, 0.001), dict(max_generations=2, quantile=0.001)),
}


@pytest.mark.parametrize("case", list(REPLAY))
def test_driver_matches_replay(ctx, mc, problem, case):
    o, target = problem
    kernel, thr, kw = REPLAY[case]
    r = mc.abc_smc(o, target, thr, 200, kernel=kernel, **kw)
    ref = replay(ctx, o, target, thr, 200, kernel, **kw)
    _same(r, ref)
    assert r["generations"] >= kw["max_generations"] - 1, r["epsilon"]
    assert r["kernel_used"][0] is None
    if case == "olcm-forced-fallback":
        assert r["kernel_used"][1:] == ["mvn"] * (r["generations"] - 1), r["kernel_used"]
    else:
        assert r["kernel_used"][1:] == [kernel] * (r["generations"] - 1), r["kernel_used"]
    print(f"{case}: eps {r['epsilon'].tolist()} simulated {r['simulated'].tolist()} used {r['kernel_used']}")


def test_driver_does_not_depend_on_chunk_size_or_gpu_count(pkg, mc, problem):
    import torch
    o, target = problem
    base = mc.abc_smc(o, target, THR, 300, max_generations=5, chunk=4096, kernel="olcm", **BOX)
    assert base["generations"] >= 3
    _same(mc.abc_smc(o, target, THR, 300, max_generations=5, chunk=512, kernel="olcm", **BOX), base, extra=())
    if torch.cuda.device_count() >= 2:
        m = pkg.MultiContext()
        try:
            _same(m.abc_smc(o, target, THR, 300, max_generations=5, chunk=4096, kernel="olcm", **BOX), base, extra=())
        finally:
            m.close()


def test_ex_component_is_abc_smc(pkg, mc, problem):
    """ecdna_b200_abc_smc_ex with the component kernel (what MultiContext.abc_smc calls) and ecdna_b200_abc_smc give
    the same bytes."""
    o, target = problem
    ex = mc.abc_smc(o, target, THR, 200, max_generations=4, kernel="component", **BOX)
    p = mc.make_params(o, 1, abc_target=np.ascontiguousarray(target, dtype=np.uint64), abc_thresholds=THR,
                       snapshots=False)
    opt = pkg.SmcOptionsT()
    opt.population, opt.quantile, opt.max_generations, opt.max_simulations = 200, 0.5, 4, 10_000_000
    opt.idx_begin = o.idx_begin
    opt.b1_range[:], opt.d0_range[:], opt.d1_range[:] = BOX["b1_range"], BOX["d0_range"], BOX["d1_range"]
    res, out = pkg.SmcResultT(), {}
    for name, dtype, tail in pkg.SMC_PARTICLE_FIELDS:
        out[name] = np.zeros((4, 200) + tail, dtype=dtype)
        setattr(res, name, out[name].ctypes.data)
    for name, dtype, tail in pkg.SMC_GENERATION_FIELDS:
        out[name] = np.zeros((4,) + tail, dtype=dtype)
        setattr(res, name, out[name].ctypes.data)
    assert pkg.lib().ecdna_b200_abc_smc(mc._h, C.byref(p), C.byref(opt), C.byref(res)) == 0
    g = int(res.generations)
    assert g == ex["generations"] and pkg.SMC_STATUS[res.status] == ex["status"]
    for k in ("idx", "parent_idx", "rates", "distance", "weight", "cells", "epsilon", "consumed", "simulated", "ess"):
        np.testing.assert_array_equal(out[k][:g].view(np.uint8), np.ascontiguousarray(ex[k]).view(np.uint8), err_msg=k)
    assert ex["kernel_used"] == [None] + ["component"] * (g - 1)
    bad = pkg.SmcKernelT(3)
    assert pkg.lib().ecdna_b200_abc_smc_ex(mc._h, C.byref(p), C.byref(opt), C.byref(bad), C.byref(res), None) == 1


# ---------------------------------------------------------------------------------------------------------------
# 7-8. the posterior, and the CLI
# ---------------------------------------------------------------------------------------------------------------
def test_posterior_matches_rejection_abc(pkg, ctx, mc, problem):
    o, target = problem
    n_rej = 1_000_000
    rates, res, ok = _rejection(pkg, ctx, o, target, 1234, 10_000_000, n_rej, TIGHT)
    acc = rates[ok][:, 1:].astype(np.float64)
    assert len(acc) >= 2000, len(acc)
    for kernel in ("mvn", "olcm"):
        r = mc.abc_smc(o, target, TIGHT, 2000, max_generations=25, max_simulations=20_000_000, kernel=kernel, **BOX)
        assert r["status"] == "reached", (kernel, r["status"], r["epsilon"])
        th, w, ess = r["rates"][-1][:, 1:].astype(np.float64), r["weight"][-1], float(r["ess"][-1])
        assert ess > 200
        for k in range(3):
            m_rej, var = acc[:, k].mean(), acc[:, k].var()
            m_smc = float(np.sum(w * th[:, k]))
            bound = 4 * np.sqrt(var / len(acc) + var / ess)
            assert abs(m_smc - m_rej) <= bound, (kernel, k, m_smc, m_rej, bound)
        print(f"{kernel}: {int(r['simulated'].sum())} draws simulated over {r['generations']} generations, ESS "
              f"{ess:.0f}, used {r['kernel_used']}")


def test_cli_kernel_option(pkg, mc, tmp_path):
    import json
    pkg.build()
    exe = os.path.join(os.path.dirname(pkg.LIB_PATH), "host", "ecdna")
    o = pkg.SimulationOptions(cells=2000, seed=7, save_snapshots=False)
    target = ob.run(oracle_opts(pkg.SimulationOptions(b0=1.0, b1=1.4, d0=0.2, d1=0.2, cells=2000, seed=7), 999),
                    hist_cap=256).hist
    tfile = tmp_path / "target.json"
    tfile.write_text(json.dumps({str(k): int(c) for k, c in enumerate(target) if c}))
    base = ["abc", "--target", str(tfile), "--generations", "4", "--population", "150", "--quantile", "0.4",
            "--max-simulations", "3000000", "--cells", "2000", "--seed", "7", "--thresholds", ",".join(map(str, THR))]
    runs = {}
    for name, extra in (("olcm", ["--kernel", "olcm"]), ("component", ["--kernel", "component"]), ("default", [])):
        out = tmp_path / name
        r = subprocess.run([exe] + base + extra + [str(out)], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        runs[name] = {f: (out / f).read_bytes() for f in sorted(os.listdir(out))}
    assert runs["default"] == runs["component"]
    res = mc.abc_smc(o, target, THR, 150, quantile=0.4, max_generations=4, max_simulations=3_000_000, kernel="olcm",
                     **BOX)
    py = tmp_path / "py"
    assert pkg.write_abc_smc(str(py), o, res) == res["generations"] >= 2
    names = sorted(os.listdir(py))
    assert sorted(runs["olcm"]) == names
    for f in names:
        assert runs["olcm"][f] == (py / f).read_bytes(), f
    js = json.loads(runs["olcm"]["abc_smc.json"])
    assert js["kernel"] == "olcm" and js["kernel_used"][0] is None and len(js["kernel_used"]) == res["generations"]
    assert "kernel" not in json.loads(runs["default"]["abc_smc.json"])
