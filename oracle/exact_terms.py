"""TEST INFRASTRUCTURE ONLY (the oracle) -- never imported by the product path.

Arbitrary-precision (mpmath) reference of every parametric term of the model description (include/gwi.h
gwi_term_kind): the per-sample log-density and its gradient with respect to the term's Lambda slots, normalisers
included.  The formulas are written from the mathematical definitions, not from the fp64 expressions of the kernels
or of oracle/popmodel.py:

  * power law          -log int_lo^hi x^alpha dx, the limit log(hi/lo) at alpha = -1   (distributions.py:100-119)
  * truncated normal   D = Phi(b) - Phi(a) from mp.ncdf                                 (distributions.py:122-143)
  * Beta               the normaliser from mp.loggamma                                  (distributions.py:146-162)
  * PL+Peak, iso+aligned (single and pair): mixtures formed from the exact components  (parametric.py:49-53,84-102)
  * low-mass window    1/(1 + exp(d/y + d/(y - d))) for EVERY y, as the reference evaluates it: a deliberate part
                       of the model definition (distributions.py:16-21), not a rounding effect

Every input is a double, taken exactly.  Gradients are analytic; ``numeric_grad`` gives mp.diff of the value for a
cross-check.

Where the reference's own fp64 formula leaves the real line, the expected result is its IEEE convention, not an
mpmath value.  Those points are named here, and an evaluation returns ``DROPPED`` (weight zero, log-density -inf):
  * outside a support: x outside [lo, hi] (power law, PL+Peak, truncated normal), x <= 0 or x >= scale (Beta, whose
    end points give 0/inf/nan), cos tilt outside [-1, 1], q outside [mmin/m1, 1] or m1 <= mmin (power law in q);
  * the window at y = 0 and y = delta (t = +inf), and wherever t > ~709.8 so that exp(t) overflows to +inf;
  * a mixture (PL+Peak, iso+aligned) whose every non-zero component is below the fp64 range.
Points too close to an fp64 range limit to have one answer (a window with t in [700, 720], a mixture whose largest
component lies in [1e-330, 1e-300], where fp64 results are subnormal) raise ``Ambiguous``: a sweep must not use them.
"""

import functools

import mpmath as mp

DPS = 50  # working precision of every evaluation (>= 40 is required; the power-law derivative near alpha = -1 cancels ~30 digits)
DROPPED = None


class Ambiguous(ValueError):
    """The point lies at an fp64 range limit where the reference's result is not well defined."""


def _m(x):
    return x if isinstance(x, mp.mpf) else mp.mpf(float(x))


def _prec():
    return mp.workdps(max(DPS, mp.mp.dps))


# ---- building blocks ------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=4096)
def _powerlaw_norm(alpha, lo, hi):
    """(-log I, d(-log I)/dalpha) with I = int_lo^hi x^alpha dx (lo, hi, alpha mp numbers)."""
    a1 = 1 + alpha
    if a1 == 0:
        L = mp.log(hi / lo)
        return -mp.log(L), -(mp.log(hi) + mp.log(lo)) / 2
    ha, la = mp.power(hi, a1), mp.power(lo, a1)
    I = (ha - la) / a1
    dI = (ha * mp.log(hi) - la * mp.log(lo)) / a1 - (ha - la) / a1**2
    return -mp.log(I), -dI / I


def _normal_interval(a, b):
    """Phi(b) - Phi(a), a < b, from mp.ncdf (in the upper tail through the identity Phi(b) - Phi(a) = Phi(-a) - Phi(-b),
    so that 1 - tiny is not formed at finite precision)."""
    if a >= 0:
        return mp.ncdf(-a) - mp.ncdf(-b)
    return mp.ncdf(b) - mp.ncdf(a)


@functools.lru_cache(maxsize=4096)
def _truncnorm_consts(mu, sig, lo, hi):
    """(log of the normaliser sigma sqrt(2 pi) D, dlog D/dmu, dlog D/dsigma) of the normal truncated to [lo, hi]."""
    a, b = (lo - mu) / sig, (hi - mu) / sig
    D = _normal_interval(a, b)
    pa, pb = mp.npdf(a), mp.npdf(b)
    return mp.log(sig) + mp.log(mp.sqrt(2 * mp.pi)) + mp.log(D), (pa - pb) / (sig * D), (a * pa - b * pb) / (sig * D)


def _truncnorm(x, mu, sig, lo, hi):
    """(log pdf, d/dmu, d/dsigma) of the normal(mu, sig) truncated to [lo, hi]."""
    lnorm, dmu_D, dsig_D = _truncnorm_consts(mu, sig, lo, hi)
    z = (x - mu) / sig
    return -z * z / 2 - lnorm, z / sig - dmu_D, z * z / sig - 1 / sig - dsig_D


def _window(d, y):
    """(S, dlog S/d delta) of the reference's window at y = x - xmin; S = 0 where its formula gives t = +inf."""
    if y == 0 or y == d:
        return mp.mpf(0), mp.mpf(0)
    t = d / y + d / (y - d)
    if 700 <= t <= 720:
        raise Ambiguous(f"window exponent t = {float(t):.6g} is at the fp64 overflow of exp")
    if t > 720:
        return mp.mpf(0), mp.mpf(0)
    S = 1 / (1 + mp.exp(t))
    return S, -(1 - S) * (1 / y + y / (y - d) ** 2)


def _mixture(parts):
    """parts: [(component value, [d component / d slot])]; -> (log sum, gradient) or DROPPED."""
    nz = [c for c, _ in parts if c != 0]
    if not nz or max(nz) < mp.mpf("1e-330"):
        return DROPPED
    if max(nz) < mp.mpf("1e-300"):
        raise Ambiguous(f"largest mixture component {mp.nstr(max(nz), 5)} is subnormal in fp64")
    tot = mp.fsum(c for c, _ in parts)
    n = len(parts[0][1])
    return mp.log(tot), [mp.fsum(dc[k] for _, dc in parts) / tot for k in range(n)]


# ---- the terms ------------------------------------------------------------------------------------------------------
# Each returns (log-density, [gradient in slot order]) or DROPPED.  Arguments are doubles.
def powerlaw(x, alpha, lo, hi):
    """POWERLAW: x^alpha / int_lo^hi; slots (alpha,)."""
    with _prec():
        x, alpha, lo, hi = map(_m, (x, alpha, lo, hi))
        if not (lo <= x <= hi):
            return DROPPED
        ln, dn = _powerlaw_norm(alpha, lo, hi)
        return alpha * mp.log(x) + ln, [mp.log(x) + dn]


def powerlaw_ratio(q, m1, beta, mmin):
    """POWERLAW_RATIO: q^beta / int_{mmin/m1}^1; slots (beta,)."""
    with _prec():
        q, m1, beta, mmin = map(_m, (q, m1, beta, mmin))
        lo = mmin / m1
        if not (lo < 1 and lo <= q <= 1):
            return DROPPED
        ln, dn = _powerlaw_norm(beta, lo, mp.mpf(1))
        return beta * mp.log(q) + ln, [mp.log(q) + dn]


def plpeak(m, alpha, mu, sig, lam, delta, mmin, mmax):
    """PLPEAK: (1 - lam) PL(m) [S(delta, m - mmin)] + lam TN(m; mu, sig, mmin, mmax); slots (alpha, mu, sig, lam[, delta]).
    delta None: no window."""
    with _prec():
        m, alpha, mu, sig, lam, mmin, mmax = map(_m, (m, alpha, mu, sig, lam, mmin, mmax))
        if not (mmin <= m <= mmax):
            return DROPPED
        ln, dn = _powerlaw_norm(alpha, mmin, mmax)
        PL = mp.exp(alpha * mp.log(m) + ln)
        S, dS = (mp.mpf(1), mp.mpf(0)) if delta is None else _window(_m(delta), m - mmin)
        ltn, dmu, dsig = _truncnorm(m, mu, sig, mmin, mmax)
        TN = mp.exp(ltn)
        A, B = (1 - lam) * PL * S, lam * TN
        gA = [A * (mp.log(m) + dn), 0, 0, -PL * S]
        gB = [0, B * dmu, B * dsig, TN]
        if delta is not None:
            gA.append(A * dS)
            gB.append(0)
        return _mixture([(A, gA), (B, gB)])


def truncnorm(x, mu, sig, lo, hi):
    """TRUNCNORM: slots (mu, sig)."""
    with _prec():
        x, mu, sig, lo, hi = map(_m, (x, mu, sig, lo, hi))
        if not (lo <= x <= hi):
            return DROPPED
        v, dmu, dsig = _truncnorm(x, mu, sig, lo, hi)
        return v, [dmu, dsig]


def beta(x, a, b, scale=1.0):
    """BETA: x^(a-1) (s-x)^(b-1) / (s^(a+b-1) B(a, b)); slots (a, b)."""
    with _prec():
        x, a, b, s = map(_m, (x, a, b, scale))
        if not (0 < x < s):
            return DROPPED
        l1, l2, ls = mp.log(x), mp.log(s - x), mp.log(s)
        lB, dA, dB = _beta_consts(a, b)
        v = (a - 1) * l1 + (b - 1) * l2 - (a + b - 1) * ls - lB
        return v, [l1 - ls - dA, l2 - ls - dB]


@functools.lru_cache(maxsize=4096)
def _beta_consts(a, b):
    """(log B(a, b), dlog B/da, dlog B/db)."""
    pab = mp.digamma(a + b)
    return mp.loggamma(a) + mp.loggamma(b) - mp.loggamma(a + b), mp.digamma(a) - pab, mp.digamma(b) - pab


def isoalign(ct, xi, sig):
    """ISOALIGN: (1 - xi)/2 + xi TN(ct; 1, sig, -1, 1); slots (xi, sig)."""
    with _prec():
        ct, xi, sig = map(_m, (ct, xi, sig))
        if not (-1 <= ct <= 1):
            return DROPPED
        ltn, _, dsig = _truncnorm(ct, mp.mpf(1), sig, mp.mpf(-1), mp.mpf(1))
        TN = mp.exp(ltn)
        return _mixture([((1 - xi) / 2, [-mp.mpf(1) / 2, 0]), (xi * TN, [TN, xi * TN * dsig])])


def isoalign_pair(ct1, ct2, xi, sig):
    """ISOALIGN_PAIR: (1 - xi)/4 + xi TN(ct1) TN(ct2); slots (xi, sig)."""
    with _prec():
        ct1, ct2, xi, sig = map(_m, (ct1, ct2, xi, sig))
        if not (-1 <= ct1 <= 1 and -1 <= ct2 <= 1):
            return DROPPED
        l1, _, d1 = _truncnorm(ct1, mp.mpf(1), sig, mp.mpf(-1), mp.mpf(1))
        l2, _, d2 = _truncnorm(ct2, mp.mpf(1), sig, mp.mpf(-1), mp.mpf(1))
        T = mp.exp(l1 + l2)
        return _mixture([((1 - xi) / 4, [-mp.mpf(1) / 4, 0]), (xi * T, [T, xi * T * (d1 + d2)])])


def smooth(x, delta, xmin=0.0, x2=None):
    """SMOOTH: log S(delta, y), y = x - xmin or x * x2 - xmin (the product taken exactly); slots (delta,)."""
    with _prec():
        y = (_m(x) if x2 is None else _m(x) * _m(x2)) - _m(xmin)
        S, dS = _window(_m(delta), y)
        if S == 0:
            return DROPPED
        return mp.log(S), [dS]


def numeric_grad(fn, args, which):
    """mp.diff of the log-density ``fn(*args)`` with respect to the arguments at positions ``which``."""
    out = []
    with _prec():
        for i in which:
            def f(t, i=i):
                a = list(args)
                a[i] = t
                return fn(*a)[0]

            out.append(mp.diff(f, _m(args[i])))
    return out


def logsumexp(values):
    """log sum exp over mp values (DROPPED entries skipped)."""
    with _prec():
        v = [x for x in values if x is not DROPPED]
        top = max(v)
        return top + mp.log(mp.fsum(mp.exp(x - top) for x in v))
