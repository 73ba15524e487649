"""CPU: both fp64 oracles (oracle/popmodel.py and, through oracle/c_oracle.py, oracle/c/gwi_oracle.c) against the
arbitrary-precision reference oracle/exact_terms.py, point by point on the sweep of tests/test_param_terms_exact.py, at
the suite's tolerances.  Also cross-checks exact_terms' analytic gradients against mp.diff of its values."""

import mpmath as mp
import numpy as np
import pytest

from oracle import c_oracle
from oracle import exact_terms as X
from oracle import popmodel
from tests import test_param_terms_exact as T


def _oracle_points(evaluate, name):
    case = T.CASES[name]
    table, _ = T.exact_table(case)
    P = case.spec.n_params
    inj = {c: np.array([p[c] for p in case.spread], dtype=np.float64) for c in case.cols}
    for i, lam in enumerate(case.lams):
        live = [j for j, r in enumerate(table[i]) if r is not X.DROPPED]
        ev = evaluate(case.spec, T._columns(case, [case.points[j] for j in live]), inj, T.TOTAL_INJ, lam)
        for e, j in enumerate(live):
            v, g = table[i][j]
            at = f"{case.name} at {case.labels[i]}, sample {case.points[j]}"
            T._check(float(ev["logBF"][e]), float(v), T.VAL_RTOL, f"{at}: log-density")
            for k in range(P):
                T._check(float(ev["J_logBF"][e, k]), float(g[k]), T.GRAD_RTOL, f"{at}: d/dLambda[{k}]")


@pytest.mark.parametrize("name", list(T.CASES))
def test_popmodel_against_exact(name):
    _oracle_points(popmodel.evaluate, name)


@pytest.mark.parametrize("name", list(T.CASES))
def test_c_oracle_against_exact(name):
    _oracle_points(c_oracle.evaluate, name)


def test_popmodel_powerlaw_derivative_at_minus_one():
    """At alpha = -1 exactly the derivative of the log-normaliser is -(log lo + log hi)/2, not 0."""
    _, d = popmodel._powerlaw_lognorm(-1.0, np.float64(3.0), np.float64(100.0))
    assert abs(d + 0.5 * (np.log(3.0) + np.log(100.0))) < 1e-15


# (function, arguments, positions of the Lambda slots among the arguments)
GRAD_POINTS = [
    (X.powerlaw, (34.0, -1.0 + 1e-7, 3.0, 100.0), (1,)),
    (X.powerlaw, (3.0, -2.35, 3.0, 100.0), (1,)),
    (X.powerlaw_ratio, (0.5, 10.0, -1.0 - 2e-9, 3.0), (2,)),
    (X.plpeak, (3.5, -2.35, 34.0, 4.5, 0.08, 1.0, 3.0, 100.0), (1, 2, 3, 4, 5)),
    (X.plpeak, (90.0, -1.0 + 1e-5, 110.0, 4.5, 0.08, None, 3.0, 100.0), (1, 2, 3, 4)),
    (X.truncnorm, (0.25, 1.7, 0.1, 0.0, 1.0), (1, 2)),
    (X.truncnorm, (0.0, -1e8, 1e8, 0.0, 1.0), (1, 2)),
    (X.beta, (1e-12, 0.05, 500.0, 1.0), (1, 2)),
    (X.beta, (0.5, 2.5, 1.0 + 1e-9, 1.0), (1, 2)),
    (X.isoalign, (0.0, 0.5, 0.1), (1, 2)),
    (X.isoalign_pair, (1.0 - 1e-6, -1.0, 1e-12, 10.0), (2, 3)),
    (X.smooth, (0.25, 0.5, 0.0), (1,)),
    (X.smooth, (3.0, 5.0, 0.0, 0.5), (1,)),
]


@pytest.mark.parametrize("fn,args,which", GRAD_POINTS, ids=[f"{f.__name__}{i}" for i, (f, _, _) in enumerate(GRAD_POINTS)])
def test_exact_gradients_match_numeric_derivatives(fn, args, which):
    _, g = fn(*args)
    num = X.numeric_grad(fn, args, which)
    with mp.workdps(X.DPS):
        for k, (a, n) in enumerate(zip(g, num)):
            assert abs(a - n) <= mp.mpf("1e-25") * max(1, abs(n)), (fn.__name__, args, k, mp.nstr(a, 30), mp.nstr(n, 30))
