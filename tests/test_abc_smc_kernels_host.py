"""The correlated ABC-SMC kernels (mvn, olcm; DESIGN.md section 9) restated in numpy and mpmath, and checked on the
CPU: the sequential-truncation density integrates to 1 over the box, the log-space tail inverse agrees with
scipy.special.ndtri_exp and mpmath, the factored log mass agrees with mpmath at 40 digits, and the OLCM closed form
equals its defining sum.  test_gpu_abc_smc_kernels.py uses these functions as its reference."""
import math

import mpmath
import numpy as np
import pytest
from scipy import integrate, special

R2 = math.sqrt(0.5)
TAIL = 5.0
TRI = {(0, 0): 0, (1, 0): 1, (1, 1): 2, (2, 0): 3, (2, 1): 4, (2, 2): 5}  # packed lower triangle (11, 21, 22, ...)


def unpack(s):
    s = np.asarray(s, dtype=np.float64)
    S = np.zeros(s.shape[:-1] + (3, 3))
    for (r, c), q in TRI.items():
        S[..., r, c] = S[..., c, r] = s[..., q]
    return S


def pack(S):
    S = np.asarray(S, dtype=np.float64)
    return np.stack([S[..., r, c] for (r, c) in TRI], axis=-1)


def free_params(ranges, cov):
    """The free parameters of the kernels: lo < hi and a variance > 0 (abc_smc.cu make_cov_args)."""
    cov = np.asarray(cov, dtype=np.float64).reshape(-1, 6)
    return [k for k in range(3) if ranges[k][0] < ranges[k][1] and np.all(cov[:, TRI[(k, k)]] > 0)]


def log_phi(x):
    """log Phi(x), finite far below the range of Phi."""
    return special.log_ndtr(x)


def log_mass(a, b):
    """log(Phi(b) - Phi(a)) for a <= b, without cancellation on either side of 0."""
    a, b = np.broadcast_arrays(np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64))
    neg = b < 0
    a2, b2 = np.where(neg, -b, a), np.where(neg, -a, b)  # mirror onto the positive side
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        xa = special.erfcx(a2 * R2)
        r = -0.5 * (b2 - a2) * (b2 + a2) + np.log(special.erfcx(b2 * R2) / xa)  # log(Phi-bar(b) / Phi-bar(a))
        tail = -0.5 * a2 * a2 + np.log(0.5 * xa) + np.log(-np.expm1(r))
        mid = np.log(special.ndtr(b2) - special.ndtr(a2))
    return np.where(a2 > 0, tail, mid)


def log_trunc_density(e, a, b, ea, be):
    """log(phi(e) sqrt(2 pi) / (Phi(b) - Phi(a))) in the factored form of the pair kernel: in a tail
    -(e - a)(e + a)/2 - log(erfcx(a/sqrt2)/2) - log1p(-Phi-bar(b)/Phi-bar(a)), with ea = e - a, be = b - e."""
    e, a, b, ea, be = np.broadcast_arrays(*[np.asarray(x, dtype=np.float64) for x in (e, a, b, ea, be)])
    neg = b < 0
    e2, a2, b2 = np.where(neg, -e, e), np.where(neg, -b, a), np.where(neg, -a, b)
    ea2, be2 = np.where(neg, be, ea), np.where(neg, ea, be)
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        xa = special.erfcx(a2 * R2)
        r = -0.5 * (ea2 + be2) * (b2 + a2) + np.log(special.erfcx(b2 * R2) / xa)
        tail = -0.5 * ea2 * (e2 + a2) - np.log(0.5 * xa) - np.log(-np.expm1(r))
        mid = -0.5 * e2 * e2 - np.log(special.ndtr(b2) - special.ndtr(a2))
    return np.where(a2 > 0, tail, mid)


def tail_inverse(T):
    """The x < -5 with log Phi(x) = T: Newton on log Phi from the asymptotic start, 4 steps (abc_smc.cu)."""
    T = np.asarray(T, dtype=np.float64)
    y = np.sqrt(-2.0 * T)
    y = np.sqrt(np.maximum(-2.0 * T - 2.0 * np.log(y) - math.log(2 * math.pi), 1.0))
    x = -y
    for _ in range(4):
        x = x - (log_phi(x) - T) * special.erfcx(-x * R2) * math.sqrt(math.pi / 2)
    return x


def trunc_normal(a, b, u):
    """N(0, 1) truncated to [a, b] from u by inverse CDF: the central case in Phi, beyond -5 (or, mirrored, +5) in
    log space."""
    a, b, u = np.broadcast_arrays(*[np.asarray(x, dtype=np.float64) for x in (a, b, u)])
    lo = b < -TAIL
    hi = a > TAIL
    aa, bb, uu = np.where(hi, -b, a), np.where(hi, -a, b), np.where(hi, 1.0 - u, u)
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        la, lb = log_phi(aa), log_phi(bb)
        T = lb + np.log(uu + (1.0 - uu) * np.exp(la - lb))
        t = np.clip(tail_inverse(np.where(lo | hi, T, -30.0)), aa, bb)
        fa, fb = special.ndtr(a), special.ndtr(b)
        mid = np.clip(special.ndtri(fa + u * (fb - fa)), a, b)  # (the kernel clamps theta to the box)
    return np.where(lo, t, np.where(hi, -t, mid))


def chol(cov, free):
    """L of Sigma over the free parameters, [..., D, D]."""
    S = unpack(cov)[..., free, :][..., :, free]
    return np.linalg.cholesky(S)


def kernel_log_density(theta, c, cov, ranges):
    """log q_c(theta) of the sequential-truncation kernel around c with Sigma = cov over the free parameters:
    sum_t log phi(e_t) - log L_tt - log(Phi(b_t) - Phi(a_t)), e = L^-1 (theta - c).  theta [n][3], c [3]."""
    free = free_params(ranges, cov)
    L = chol(np.asarray(cov, dtype=np.float64).reshape(6), free)
    x = np.atleast_2d(np.asarray(theta, dtype=np.float64))[:, free]
    d = x - np.asarray(c, dtype=np.float64)[free]
    e = np.linalg.solve(L, d.T).T
    out = np.zeros(len(x))
    for t, k in enumerate(free):
        lo, hi = ranges[k]
        s = L[t, t]
        m = x[:, t] - s * e[:, t]
        out += -0.5 * e[:, t] ** 2 - 0.5 * math.log(2 * math.pi) - math.log(s) - log_mass((lo - m) / s, (hi - m) / s)
    return out


def rosenblatt(theta, c, cov, ranges):
    """(Phi(e_t) - Phi(a_t)) / (Phi(b_t) - Phi(a_t)) per free coordinate, in log space: the uniforms that drew theta.
    Returns (u [n][D], e, a, b, L)."""
    free = free_params(ranges, cov)
    L = chol(np.asarray(cov, dtype=np.float64).reshape(6), free)
    x = np.atleast_2d(np.asarray(theta, dtype=np.float64))[:, free]
    d = x - np.asarray(c, dtype=np.float64)[free]
    e = np.linalg.solve(L, d.T).T
    a, b = np.zeros_like(e), np.zeros_like(e)
    for t, k in enumerate(free):
        lo, hi = ranges[k]
        m = x[:, t] - L[t, t] * e[:, t]
        a[:, t], b[:, t] = (lo - m) / L[t, t], (hi - m) / L[t, t]
    e = np.clip(e, a, b)
    with np.errstate(divide="ignore", invalid="ignore"):
        up = a > 0  # on the positive side: 1 - u = (Phi-bar(e) - Phi-bar(b)) / (Phi-bar(a) - Phi-bar(b))
        num = np.where(up, log_mass(e, b), log_mass(a, e))
        u = np.exp(num - log_mass(a, b))
        u = np.where(up, 1.0 - u, u)
    return u, e, a, b, L


def olcm_closed_form(theta, w, sel, j):
    """Sigma_j = C + (m - theta_j)(m - theta_j)^T over the selected particles, weights renormalised."""
    ws = w[sel] / w[sel].sum()
    m = ws @ theta[sel]
    d = theta[sel] - m
    C = (ws[:, None] * d).T @ d
    v = m - theta[j]
    return C + np.outer(v, v)


# ---------------------------------------------------------------------------------------------------------------
BOX = [(1.0, 2.0), (0.0, 0.5), (0.0, 0.5)]


def _corr_cov(sd, rho):
    """Sigma from sds and the correlations (r12, r13, r23)."""
    R = np.array([[1, rho[0], rho[1]], [rho[0], 1, rho[2]], [rho[1], rho[2], 1]], dtype=np.float64)
    return pack(np.outer(sd, sd) * R)


@pytest.mark.parametrize("where, c", [("interior", (1.4, 0.2, 0.25)), ("edge", (1.3, 0.0, 0.2)),
                                      ("corner", (1.0, 0.0, 0.0))])
def test_density_integrates_to_one(where, c):
    """Two free parameters (b1 fixed) with correlation 0.9 over the box, and all three for the interior parent."""
    cov = _corr_cov([0.3, 0.12, 0.1], [0.0, 0.0, 0.9])
    fixed = [(1.0, 1.0), BOX[1], BOX[2]]
    c2 = (1.0,) + tuple(c[1:])
    f2 = lambda y, z: math.exp(kernel_log_density([[1.0, y, z]], c2, cov, fixed)[0])  # noqa: E731
    tot, err = integrate.nquad(f2, [BOX[1], BOX[2]], opts={"epsabs": 1e-10, "epsrel": 1e-8})
    assert abs(tot - 1.0) < 1e-6, (where, tot, err)
    if where == "interior":
        cov = _corr_cov([0.3, 0.12, 0.1], [-0.6, 0.3, 0.5])
        f3 = lambda x, y, z: math.exp(kernel_log_density([[x, y, z]], c, cov, BOX)[0])  # noqa: E731
        tot3, err3 = integrate.nquad(f3, BOX, opts={"epsabs": 1e-5, "epsrel": 1e-4, "limit": 10})
        assert abs(tot3 - 1.0) < 1e-3, (tot3, err3)


def _mp_trunc_inverse(a, b, u):
    """e with (Phi(e) - Phi(a)) / (Phi(b) - Phi(a)) = u, at 60 digits."""
    with mpmath.workdps(60):
        a, b, u = mpmath.mpf(a), mpmath.mpf(b), mpmath.mpf(u)
        if a > 0:  # the upper tail, in Phi-bar
            pb = lambda x: mpmath.erfc(x / mpmath.sqrt(2)) / 2  # noqa: E731
            target = pb(a) - u * (pb(a) - pb(b))
            return float(mpmath.findroot(lambda x: mpmath.log(pb(x)) - mpmath.log(target), (a + b) / 2))
        ph = mpmath.ncdf
        target = ph(a) + u * (ph(b) - ph(a))
        return float(mpmath.findroot(lambda x: mpmath.log(ph(x)) - mpmath.log(target), (a + b) / 2))


@pytest.mark.parametrize("a", [0.0, 5.0, 37.0, 1e2, 1e3, 1e4])
def test_tail_inverse(a):
    """Intervals [a, a + 3/a] (0: [0, 3]) and, mirrored, [-a - 3/a, -a]: the sampler against mpmath, and the Newton
    inverse of log Phi against scipy.special.ndtri_exp."""
    w = 3.0 / a if a else 3.0
    us = np.array([0.0, 1e-12, 0.01, 0.3, 0.5, 0.77, 0.99, 1 - 2.0 ** -53])
    for lo, hi, sign in ((a, a + w, 1.0), (-a - w, -a, -1.0)):
        got = trunc_normal(lo, hi, us)
        assert np.all((got >= lo) & (got <= hi)) and np.all(np.isfinite(got))
        for u, g in zip(us, got):
            ref = _mp_trunc_inverse(lo, hi, u)
            # 4 ulp of the result, plus in the central case the rounding of the target Phi(a) + u (Phi(b) - Phi(a)) in f64
            # carried through the inverse (divided by the density phi at the result)
            tol = 4 * np.spacing(abs(ref))
            if not (hi < -5 or lo > 5):
                tol += 4 * 2.0 ** -53 * special.ndtr(hi) / max(math.exp(-ref * ref / 2) / math.sqrt(2 * math.pi), 1e-300)
            assert abs(g - ref) <= tol, (lo, hi, u, g, ref)
    T = -np.logspace(math.log10(15.5), 9, 200)  # (log Phi(-5) = -15.06)
    np.testing.assert_allclose(tail_inverse(T), special.ndtri_exp(T), rtol=1e-12, atol=0)


def test_factored_log_mass_against_mpmath():
    cases = []
    for a in (-3.0, -0.4, 0.0, 0.2, 2.0, 5.0, 37.0, 100.0, 1e4, 1e6):
        for width in (1e-6, 0.01, 1.0, 50.0):
            for f in (0.0, 0.3, 1.0):
                cases.append((a, a + width, f * width))
                cases.append((-a - width, -a, f * width))
    for a, b, ea in cases:
        e = a + ea
        be = b - e
        got = float(log_trunc_density(e, a, b, ea, be))
        lm = float(log_mass(a, b))
        with mpmath.workdps(40):
            A, B, E = mpmath.mpf(a), mpmath.mpf(b), mpmath.mpf(a) + mpmath.mpf(ea)
            mass = mpmath.ncdf(B) - mpmath.ncdf(A) if b <= 0 or a < 0 else \
                (mpmath.erfc(A / mpmath.sqrt(2)) - mpmath.erfc(B / mpmath.sqrt(2))) / 2
            ref_lm = mpmath.log(mass)
            Bd = E + mpmath.mpf(be)  # (the interval the density sees: e - a and b - e exact, as edge distances are)
            mass_d = mpmath.ncdf(Bd) - mpmath.ncdf(A) if Bd <= 0 or a < 0 else \
                (mpmath.erfc(A / mpmath.sqrt(2)) - mpmath.erfc(Bd / mpmath.sqrt(2))) / 2
            ref = -E * E / 2 - mpmath.log(mass_d)
        # f64 relative error on the magnitudes involved, and the conditioning of a narrow interval's mass (relative
        # error of a few ulp in erfcx or Phi, over 1 - Phi-bar(b) / Phi-bar(a) ~ (b - a) max(1, |a|))
        cond = 1.0 + 1.0 / ((b - a) * max(1.0, min(abs(a), abs(b))))
        scale = 1.0 + abs(float(ref)) + abs(a) * (b - a)
        assert abs(got - float(ref)) <= 1e-13 * scale + 4e-15 * cond, (a, b, ea, got, float(ref))
        assert abs(lm - float(ref_lm)) <= 1e-13 * (1.0 + abs(float(ref_lm))) + 4e-15 * cond, (a, b, lm, float(ref_lm))


def test_olcm_closed_form_is_the_defining_sum():
    rng = np.random.default_rng(5)
    M = 400
    theta = np.column_stack([rng.uniform(1, 2, M), rng.uniform(0, 0.5, M), rng.uniform(0, 0.5, M)])
    theta[:, 2] = 0.5 * theta[:, 2] + 0.3 * theta[:, 1]
    w = rng.uniform(0.1, 1, M)
    w /= w.sum()
    sel = rng.uniform(size=M) < 0.4
    ws = w[sel] / w[sel].sum()
    for j in (0, 7, 123, 399):
        brute = sum(wk * np.outer(tk - theta[j], tk - theta[j]) for wk, tk in zip(ws, theta[sel]))
        np.testing.assert_allclose(olcm_closed_form(theta, w, sel, j), brute, rtol=1e-12, atol=1e-15)


def test_sampler_and_rosenblatt_are_inverse():
    """The numpy sampler drawn from u returns u through the Rosenblatt transform, across central and tail cases."""
    rng = np.random.default_rng(9)
    for a, b in ((-1.0, 2.0), (-40.0, -6.0), (6.0, 7.0), (-3.0, -2.0), (37.0, 37.1), (-1e4 - 1e-3, -1e4)):
        u = rng.uniform(size=1000)
        e = trunc_normal(a, b, u)
        assert np.all((e >= a) & (e <= b))
        with np.errstate(divide="ignore"):
            back = np.where(a > 0, 1.0 - np.exp(log_mass(e, b) - log_mass(a, b)), np.exp(log_mass(a, e) - log_mass(a, b)))
        np.testing.assert_allclose(back, u, atol=1e-9 * max(1.0, abs(a)) * 100)
