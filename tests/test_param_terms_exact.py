"""GPU (-m gpu): every parametric term of the model description against an arbitrary-precision reference.

The stream-kernel tests prove the kernels' index arithmetic and accumulators against oracle/popmodel.py, which uses the
same closed forms as the kernels: where a formula loses precision both lose it together.  Here each term kind is the
only term of a ``spec.ModelSpec`` built on a hand-made catalog in which every event holds ONE sample, so that
``logBF_i`` is the term's log-density at x_i and ``J_logBF_i`` its gradient, and each is compared with
oracle/exact_terms.py (mpmath) point by point.  The injection set is the same points plus a seeded spread of 200 more;
``log_mu`` and ``J_log_mu`` are compared with an mpmath log-sum-exp of the exact values.  The parameters sweep fixed
lists that reach the edges: the power law within 1e-15 of alpha = -1, truncated normals up to 30 sigma outside their
range and sigma up to 1e8, Beta shapes from 0.05 to 500, the window at and around its poles.  Finally each term's whole
parameter list runs as one ``loglike_batch`` (one chain per Lambda), which checks the per-chain constants of the
prologue at the same edge values.

Tolerances are the suite's, per point: values |d| <= 1e-10 max(1, |exact|), each gradient component
|d| <= 1e-8 max(1, |exact|).  Points where the reference's own fp64 formula gives zero weight (outside a support, the
window's poles, a mixture whose every component underflows) must give zero weight; exact_terms names them.
tests/test_param_terms_exact_emulated.py runs the same tests on the host warp emulator.
"""

import mpmath as mp
import numpy as np
import pytest

from gwinferno_b200 import capi
from gwinferno_b200 import spec as S
from oracle import exact_terms as X
from oracle import popmodel

pytestmark = pytest.mark.gpu

VAL_RTOL, GRAD_RTOL = 1e-10, 1e-8
TOTAL_INJ = 1000.0
N_SPREAD = 200


def up(x):
    return float(np.nextafter(x, np.inf))


def down(x):
    return float(np.nextafter(x, -np.inf))


ALPHA_BAND = sorted({-1.0} | {-1.0 + s * d for s in (1.0, -1.0) for d in (1e-15, 1e-12, 5e-10, 1e-9, 2e-9, 1e-8, 1e-7, 1e-6, 1e-5, 1e-4, 1e-3, 1e-2)})
ALPHAS = ALPHA_BAND + [-12.0, -4.0, -2.35, 0.0, 3.0, 12.0]


class Case:
    """One term kind: its model, the sample points (dicts column -> value), the Lambda list and the exact reference
    ``exact(lam, point)``."""

    def __init__(self, name, term, n_params, points, lams, exact, spread, labels=None):
        self.name, self.points, self.lams, self.exact, self.spread = name, points, [np.asarray(l, dtype=float) for l in lams], exact, spread
        self.spec = S.ModelSpec([term], [], [], n_params)
        self.cols = list(term.cols)
        self.labels = labels or [str(list(l)) for l in self.lams]


def _spread(rng, **ranges):
    return [{c: float(rng.uniform(*r)) for c, r in ranges.items()} for _ in range(N_SPREAD)]


def case_powerlaw():
    lo, hi = 3.0, 100.0
    pts = [{"x": v} for v in (lo, up(lo), 34.0, hi, down(lo), up(hi))]
    return Case("POWERLAW", S.Term(S.TERM_POWERLAW, ["x"], slots=[0], cst=[lo, hi]), 1, pts, [[a] for a in ALPHAS],
                lambda lam, p: X.powerlaw(p["x"], lam[0], lo, hi), _spread(np.random.default_rng(1), x=(lo, hi)))


def case_powerlaw_ratio():
    mmin = 3.0
    pts = []
    for m1 in (3.0 * (1.0 + 1e-6), 3.5, 10.0, 50.0, 100.0):
        qlo = mmin / m1
        pts += [{"q": up(qlo), "m1": m1}, {"q": 0.5 * (qlo + 1.0), "m1": m1}, {"q": 1.0, "m1": m1}]
    pts += [{"q": down(mmin / 10.0), "m1": 10.0}, {"q": up(1.0), "m1": 10.0}, {"q": 0.9, "m1": mmin}, {"q": 0.9, "m1": 2.0}]
    rng = np.random.default_rng(2)
    spread = []
    for _ in range(N_SPREAD):
        m1 = float(rng.uniform(3.2, 100.0))
        spread.append({"q": float(rng.uniform(mmin / m1, 1.0)), "m1": m1})
    return Case("POWERLAW_RATIO", S.Term(S.TERM_POWERLAW_RATIO, ["q", "m1"], slots=[0], cst=[mmin]), 1, pts, [[b] for b in ALPHAS],
                lambda lam, p: X.powerlaw_ratio(p["q"], p["m1"], lam[0], mmin), spread)


def case_truncnorm(lo, hi):
    pts = [{"x": v} for v in (lo, up(lo), 0.5 * (lo + hi) + 0.125, hi, down(lo), up(hi))]
    lams = []
    for sig in (1e-3, 0.1, 1.0, 1e3, 1e6, 1e8):
        mus = [0.5 * (lo + hi) + 0.1 * (hi - lo), lo, hi] + [b + s * k * sig for k in (1, 3, 5, 6, 8, 12, 20, 30) for b, s in ((lo, -1.0), (hi, 1.0))]
        lams += [[mu, sig] for mu in mus]
    return Case(f"TRUNCNORM[{lo:g},{hi:g}]", S.Term(S.TERM_TRUNCNORM, ["x"], slots=[0, 1], cst=[lo, hi]), 2, pts, lams,
                lambda lam, p: X.truncnorm(p["x"], lam[0], lam[1], lo, hi), _spread(np.random.default_rng(3), x=(lo, hi)))


def case_plpeak(windowed):
    mmin, mmax = 3.0, 100.0
    base = dict(alpha=-2.35, mu=34.0, sig=4.5, lam=0.08, delta=1.0)
    keys = ("alpha", "mu", "sig", "lam") + (("delta",) if windowed else ())
    variants = [dict(base, alpha=a) for a in ALPHAS]
    if windowed:
        variants += [dict(base, mu=mu) for mu in (34.0, mmin, mmax) + tuple(b + s * k * base["sig"] for k in (1, 5, 20) for b, s in ((mmin, -1.0), (mmax, 1.0)))]
        variants += [dict(base, sig=s) for s in (0.05, 50.0)] + [dict(base, sig=0.05, mu=mu) for mu in (mmin - 20 * 0.05, mmax + 20 * 0.05)]
        variants += [dict(base, lam=l) for l in (0.0, 1e-6, 1.0)] + [dict(base, delta=d) for d in (0.01, 8.0)]
    deltas = (0.01, 1.0, 8.0) if windowed else (1.0,)
    ms = sorted({mmin, 34.0, mmax} | {v for d in deltas for v in (mmin + d / 2, mmin + d)} | {up(mmin)})
    pts = [{"m": m} for m in ms] + [{"m": down(mmin)}, {"m": up(mmax)}]
    term = S.Term(S.TERM_PLPEAK, ["m"], slots=[0, 1, 2, 3, 4 if windowed else -1], cst=[mmin, mmax])
    labels = [", ".join(f"{k}={v[k]!r}" for k in keys) for v in variants]
    return Case("PLPEAK" + ("+window" if windowed else ""), term, len(keys), pts, [[v[k] for k in keys] for v in variants],
                lambda lam, p: X.plpeak(p["m"], lam[0], lam[1], lam[2], lam[3], lam[4] if windowed else None, mmin, mmax),
                _spread(np.random.default_rng(4), m=(mmin, mmax)), labels)


CT = (-1.0, up(-1.0), 0.0, 1.0 - 1e-6, 1.0)
# the spread stays where the aligned component of sigma = 0.01 is far above the fp64 range
ISO_SPREAD = (0.9, 1.0)
ISO_LAMS = [[xi, sig] for xi in (0.0, 1e-12, 0.5, 1.0) for sig in (0.01, 0.1, 1.0, 10.0, 1e3)]


def case_isoalign():
    pts = [{"ct": c} for c in CT] + [{"ct": down(-1.0)}, {"ct": up(1.0)}]
    return Case("ISOALIGN", S.Term(S.TERM_ISOALIGN, ["ct"], slots=[0, 1]), 2, pts, ISO_LAMS,
                lambda lam, p: X.isoalign(p["ct"], lam[0], lam[1]), _spread(np.random.default_rng(5), ct=ISO_SPREAD))


def case_isoalign_pair():
    pts = [{"c1": a, "c2": b} for a in CT for b in (CT[0], CT[2], CT[4])] + [{"c1": 0.0, "c2": up(1.0)}]
    return Case("ISOALIGN_PAIR", S.Term(S.TERM_ISOALIGN_PAIR, ["c1", "c2"], slots=[0, 1]), 2, pts, ISO_LAMS,
                lambda lam, p: X.isoalign_pair(p["c1"], p["c2"], lam[0], lam[1]), _spread(np.random.default_rng(6), c1=ISO_SPREAD, c2=ISO_SPREAD))


def case_beta():
    shapes = (0.05, 0.5, 1.0, 1.0 + 1e-9, 2.5, 50.0, 500.0)
    pts = [{"x": v} for v in (1e-300, 1e-12, 0.5, 1.0 - 1e-12, 0.0, 1.0)]
    return Case("BETA", S.Term(S.TERM_BETA, ["x"], slots=[0, 1], cst=[1.0]), 2, pts, [[a, b] for a in shapes for b in shapes],
                lambda lam, p: X.beta(p["x"], lam[0], lam[1], 1.0), _spread(np.random.default_rng(7), x=(0.05, 0.95)))


SMOOTH_DELTAS = (1e-3, 0.5, 5.0, 20.0)


def case_smooth(product):
    ys = sorted({1e-6, 100.0} | {v for d in SMOOTH_DELTAS for v in (d / 2, d * (1 - 1e-9), d, d * (1 + 1e-9), 2 * d)} | {0.0})
    # col0 * col1 with col1 = 0.5: the product is exact, so both sides see the same y
    pts = [{"y": 2.0 * y, "w": 0.5} for y in ys] if product else [{"y": y} for y in ys]
    term = S.Term(S.TERM_SMOOTH, ["y", "w"] if product else ["y"], slots=[0], cst=[0.0])
    rng = np.random.default_rng(8)
    spread = [dict(y=float(rng.uniform(25.0, 200.0)) * (2.0 if product else 1.0), **({"w": 0.5} if product else {})) for _ in range(N_SPREAD)]
    return Case("SMOOTH" + ("[col0*col1]" if product else "[col0]"), term, 1, pts, [[d] for d in SMOOTH_DELTAS],
                lambda lam, p: X.smooth(p["y"], lam[0], 0.0, p.get("w")), spread)


CASES = {c.name: c for c in (case_powerlaw(), case_powerlaw_ratio(), case_truncnorm(0.0, 1.0), case_truncnorm(-1.0, 1.0), case_plpeak(False),
                              case_plpeak(True), case_isoalign(), case_isoalign_pair(), case_beta(), case_smooth(False), case_smooth(True))}


# ---- exact values ---------------------------------------------------------------------------------------------------
_TABLES = {}


def exact_table(case):
    """Exact results of every (Lambda, point) and (Lambda, spread point): lists [lam][point] of X results."""
    if case.name not in _TABLES:
        _TABLES[case.name] = _exact_table(case)
    return _TABLES[case.name]


def _exact_table(case):
    pts = [case.exact(lam, p) for lam in case.lams for p in case.points]
    spr = [case.exact(lam, p) for lam in case.lams for p in case.spread]
    n, s = len(case.points), len(case.spread)
    return [pts[i * n : (i + 1) * n] for i in range(len(case.lams))], [spr[i * s : (i + 1) * s] for i in range(len(case.lams))]


def exact_injections(res, P):
    """log mu, J_log mu, log N_eff,inj and J_log N_eff,inj of the injection set from exact per-point results."""
    with mp.workdps(X.DPS):
        live = [r for r in res if r is not X.DROPPED]
        top = max(v for v, _ in live)
        w = [mp.exp(v - top) for v, _ in live]
        S1, S2 = mp.fsum(w), mp.fsum(x * x for x in w)
        G1 = [mp.fsum(wi * g[k] for wi, (_, g) in zip(w, live)) for k in range(P)]
        G2 = [mp.fsum(wi * wi * g[k] for wi, (_, g) in zip(w, live)) for k in range(P)]
        N = mp.mpf(TOTAL_INJ)
        den = S2 - S1 * S1 / N
        log_mu = top + mp.log(S1) - mp.log(N)
        J_mu = [g / S1 for g in G1]
        ln_inj = 2 * mp.log(S1) - mp.log(den)
        J_inj = [2 * G1[k] / S1 - (2 * G2[k] - 2 * S1 * G1[k] / N) / den for k in range(P)]
        return float(log_mu), np.array([float(x) for x in J_mu]), float(ln_inj), np.array([float(x) for x in J_inj])


def _check(got, want, rtol, what):
    err = abs(got - want) / max(1.0, abs(want))
    assert err <= rtol, f"{what}: got {got!r}, exact {want!r}, |d|/max(1,|exact|) = {err:.3g} > {rtol:g}"
    return err


def _columns(case, points):
    return {c: np.array([[p[c]] for p in points], dtype=np.float64) for c in case.cols}


def _inj_columns(case):
    allp = case.points + case.spread
    return {c: np.array([p[c] for p in allp], dtype=np.float64) for c in case.cols}


# ---- the tests ------------------------------------------------------------------------------------------------------
def run_points(case, worst):
    """Model.evaluate per Lambda: every finite point as a one-sample event, the zero-weight points and the spread in the
    injection set."""
    table, spread = exact_table(case)
    P = case.spec.n_params
    inj = _inj_columns(case)
    groups = {}
    for i in range(len(case.lams)):
        live = tuple(j for j, r in enumerate(table[i]) if r is not X.DROPPED)
        assert live, f"{case.name} {case.labels[i]}: no finite point"
        groups.setdefault(live, []).append(i)
    for live, lam_idx in groups.items():
        cat = capi.Catalog(_columns(case, [case.points[j] for j in live]), inj, TOTAL_INJ)
        mdl = capi.Model(cat, case.spec)
        try:
            for i in lam_idx:
                lam, where = case.lams[i], f"{case.name} at {case.labels[i]}"
                r = mdl.evaluate(lam)
                for e, j in enumerate(live):
                    v, g = table[i][j]
                    at = f"{where}, sample {case.points[j]}"
                    worst["value"] = max(worst["value"], _check(float(r["logBF"][e]), float(v), VAL_RTOL, f"{at}: log-density"))
                    for k in range(P):
                        worst["gradient"] = max(worst["gradient"], _check(float(r["J_logBF"][e, k]), float(g[k]), GRAD_RTOL, f"{at}: d/dLambda[{k}]"))
                log_mu, J_mu, _, _ = exact_injections(table[i] + spread[i], P)
                worst["value"] = max(worst["value"], _check(r["log_mu"], log_mu, VAL_RTOL, f"{where}: log_mu"))
                for k in range(P):
                    worst["gradient"] = max(worst["gradient"], _check(float(r["J_log_mu"][k]), float(J_mu[k]), GRAD_RTOL, f"{where}: J_log_mu[{k}]"))
        finally:
            mdl.close()
            cat.close()


def run_batch(case, worst):
    """The whole Lambda list as one loglike_batch: one chain per Lambda, events = the points finite at every Lambda,
    Nobs = their count, marginalize_selection on, the N_eff and variance cuts off (one-sample events have N_eff = 1)."""
    table, spread = exact_table(case)
    P = case.spec.n_params
    live = [j for j in range(len(case.points)) if all(t[j] is not X.DROPPED for t in table)]
    E = len(live)
    cat = capi.Catalog(_columns(case, [case.points[j] for j in live]), _inj_columns(case), TOTAL_INJ)
    mdl = capi.Model(cat, case.spec, need_neff_grad=True)
    try:
        ll, gg, head = mdl.loglike_batch(np.stack(case.lams), E, marginalize_selection=True, min_neff_cut=False)
    finally:
        mdl.close()
        cat.close()
    for i, lam in enumerate(case.lams):
        where = f"{case.name} chain {i} at {case.labels[i]}"
        v = np.array([float(table[i][j][0]) for j in live])
        J = np.array([[float(x) for x in table[i][j][1]] for j in live])
        log_mu, J_mu, ln_inj, J_inj = exact_injections(table[i] + spread[i], P)
        ev = dict(logBF=v, logNeff=np.zeros(E), var=np.zeros(E), log_mu=log_mu, logNeff_inj=ln_inj, var_inj=np.exp(-ln_inj) - 1.0 / TOTAL_INJ,
                  J_logBF=J, J_log_mu=J_mu, J_logNeff_inj=J_inj)
        l_x, g_x, _ = popmodel.hierarchical_log_likelihood(ev, E, marginalize_selection=True, min_neff_cut=False)
        assert head[i, 1] == 1.0 and head[i, 7] == 0.0, (where, head[i])
        # a sum of E + 1 terms: its rounding scales with the sum of their magnitudes
        scale = np.sum(np.abs(v)) + E * abs(log_mu) + E * (3 + E) / 2 * np.exp(-ln_inj)
        worst["value"] = max(worst["value"], _check(ll[i], l_x, VAL_RTOL * max(1.0, scale) / max(1.0, abs(l_x)), f"{where}: log L"))
        gscale = np.sum(np.abs(J), axis=0) + E * np.abs(J_mu) + E * (3 + E) / 2 * np.exp(-ln_inj) * np.abs(J_inj)
        for k in range(P):
            _check(gg[i, k], g_x[k], GRAD_RTOL * max(1.0, gscale[k]) / max(1.0, abs(g_x[k])), f"{where}: d log L/dLambda[{k}]")


WORST = {}


@pytest.mark.parametrize("name", list(CASES))
def test_term_points(name):
    w = WORST.setdefault(name, {"value": 0.0, "gradient": 0.0})
    run_points(CASES[name], w)
    print(f"{name}: worst per-point error: value {w['value']:.3g}, gradient {w['gradient']:.3g}")


@pytest.mark.parametrize("name", list(CASES))
def test_term_batch(name):
    run_batch(CASES[name], WORST.setdefault(name, {"value": 0.0, "gradient": 0.0}))
