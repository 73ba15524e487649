"""GPU (-m gpu): every stream-kernel instantiation the library can launch, against the fp64 oracle.

The two stream kernels are templates (stream.cuh: one-role kernel <NS, NDEEP, NLIN | PARAM, G2> and a max-only
pass per NS; stream_cta.cuh: CTA-cooperative kernel <NS, NDEEP, NLIN>), and which instantiation runs depends on the
model and on the plan.  The models here are ``spec.ModelSpec`` objects built directly on a seeded synthetic catalog
(8 coordinate columns and a sampling prior; ragged events of 1 .. 2000 samples, 2e4 injections), one per (number of
spline dims, non-spline terms), and every model runs through every geometry it admits: both kernels, every deep-dim
count, with and without the N_eff moments, several chunk lengths and both plan builders.  Each run reads back the
geometry that actually ran, derives its instantiation key with the rule of api.cu and checks values, Jacobians, the
likelihood and its gradient, the exact-shift path and a 3-chain batch against oracle/popmodel.py.  The last matrix
test asserts that every key the pick tables can return ran at least once.  The limits of the model description
(8 spline dims, 64 default-knot splines, 61 knot pieces), shared-memory pressure and the device plan builder's
host fallback are checked on both sides of each limit.

Tolerances are the suite's: values 1e-10 relative, Jacobians and gradients 1e-8; at the wide coefficient scale
(~3) the 1e-9 / 1e-7 of test_gpu_parity.test_wide_coefficient_range_shift_bound.
tests/test_kernel_matrix_emulated.py runs the same tests on the host warp emulator (a subset by default).
"""

import json
import os

import numpy as np
import pytest

from gwinferno_b200 import capi
from gwinferno_b200 import spec as S
from oracle import popmodel

pytestmark = pytest.mark.gpu

VAL_RTOL, GRAD_RTOL = 1e-10, 1e-8
WIDE_VAL_RTOL, WIDE_GRAD_RTOL = 1e-9, 1e-7
MAX_SPLINE_DIMS = 8  # gwi_internal.h MAX_SPLINE_DIMS
MAXLIN = 2  # stream.cuh MAXLIN: register-resident linear terms
MAX_DEEP = 4  # GWI_PICK / GWI_PICK_CTA instantiate NDEEP <= min(NS, 4)
EVENT_SIZES = (1, 2, 37, 300, 2000, 2, 37, 1)
N_INJ = 20000
TOTAL_INJ = 50000.0
CHUNK_STEPS = (0, 2, 4, 6, 32)  # CTA chunks shorter than, equal to and longer than the 4-stage ring
MODES = ("lin0", "lin1", "lin2", "lin3", "param", "dens")
SMALL_SPLINES = (12, 4, 9, 6, 7, 5, 10, 8)  # small enough for every deep-dim count with the N_eff moments
LARGE_SPLINES = (40, 23, 64, 17, 5, 31, 9, 50)


# ---- the instantiation tables of the pick functions, mirrored -------------------------------------------------------
def one_role_keys():
    """stream.cuh pick_stream_for_ns: NDEEP 0..min(NS, 4); nlin 0..2 register-resident or the generic loop; G2."""
    return {("one", ns, nd, v, g2) for ns in range(MAX_SPLINE_DIMS + 1) for nd in range(min(ns, MAX_DEEP) + 1) for v in (0, 1, 2, "P") for g2 in (False, True)}


def cta_keys():
    """stream_cta.cuh pick_stream_cta_for_ns: NS 1..8, NDEEP 1..min(NS, 4), NLIN 0..2 (no G2, no generic loop)."""
    return {("cta", ns, nd, nl) for ns in range(1, MAX_SPLINE_DIMS + 1) for nd in range(1, min(ns, MAX_DEEP) + 1) for nl in range(MAXLIN + 1)}


def max_keys():
    """The max-only pass of the one-role kernel (one per NS) and stream_cta_max_kernel."""
    return {("max", ns) for ns in range(MAX_SPLINE_DIMS + 1)} | {("ctamax",)}


# keys of the tables that no model description can select
UNREACHABLE = {
    ("one", 0, 0, 0, False): "no spline dim and no non-spline term leaves no parameter: the library refuses n_params = 0",
    ("one", 0, 0, 0, True): "no spline dim and no non-spline term leaves no parameter: the library refuses n_params = 0",
}


def instantiation_key(info, plan0, g2, density):
    """The kernel that ran, from what the model reports (api.cu: a generic term or a spline density selects the PARAM
    variant, which then handles every non-spline term; otherwise up to MAXLIN linear terms are register-resident)."""
    ns, nd, nlin, npar = info["n_spline_dims"], info["n_deep"], info["n_linear"], info["n_param_terms"]
    lw = int(plan0[10])  # warps that share a chunk: > 1 only in the CTA-cooperative kernel
    if info["active_switches"] & 4:
        assert lw >= 2 and info["block_threads"] == 32 * (lw + nd)
        return ("cta", ns, nd, nlin)
    assert lw == 1 and info["block_threads"] % 32 == 0 and 32 <= info["block_threads"] <= 256
    param = nlin + npar > min(nlin, MAXLIN) or density
    return ("one", ns, nd, "P" if param else min(nlin, MAXLIN), bool(g2))


# ---- models ---------------------------------------------------------------------------------------------------------
def catalog_columns(seed, sizes=EVENT_SIZES, n_inj=N_INJ, n_cols=MAX_SPLINE_DIMS):
    """Columns c0 .. c{n_cols-1} in [1, 10] and a sampling prior.  Events of one or two samples lie inside every range
    of the models, so that each event keeps a finite log BF and the likelihood passes its cuts."""
    rng = np.random.default_rng(seed)

    def draw(n, inside):
        lo, hi = (2.0, 8.0) if inside else (1.0, 10.0)
        d = {f"c{k}": rng.uniform(lo, hi, n) for k in range(n_cols)}
        d["prior"] = rng.uniform(0.5, 2.0, n)
        return d

    src = {True: draw(sum(s for s in sizes if s <= 2), True), False: draw(sum(s for s in sizes if s > 2), False)}
    used = {True: 0, False: 0}
    pe = {k: [] for k in src[True]}
    for s in sizes:
        o = used[s <= 2]
        for k in pe:
            pe[k].append(src[s <= 2][k][o : o + s])
        used[s <= 2] += s
    return pe, draw(n_inj, False)


def explicit_knots(xi_lo, xi_hi, degree, n_inner, repeat=True):
    """Knot vector in spline-coordinate units: ``n_inner`` uniform knots on [xi_lo, xi_hi] (one interior knot repeated
    if ``repeat``) extended by ``degree`` knots on either side.  Returns (knots, n_splines)."""
    k = degree + 1
    inner = np.linspace(xi_lo, xi_hi, n_inner)
    if repeat:
        inner = np.sort(np.concatenate([inner, [inner[n_inner // 2]]]))
    dx = (xi_hi - xi_lo) / (n_inner - 1)
    t = np.concatenate([xi_lo - dx * np.arange(k - 1, 0, -1), inner, xi_hi + dx * np.arange(1, k)])
    return t, t.size - k


def knot_pieces(t, x0, x1):
    """Polynomial pieces of a knot vector over [x0, x1] as plan.cpp build_piece_table counts them: every span of
    positive length that meets the range (half-open spans: one that starts at x1 counts), plus one piece below the
    first knot and one at / beyond the last knot if those lie inside the range."""
    n = int(t[0] > x0) + int(t[-1] <= x1)
    return n + sum(1 for a, b in zip(t[:-1], t[1:]) if b - a > 0 and b > x0 and a <= x1)


class Model:
    """A ModelSpec and the Lambda layout it was built with."""

    def __init__(self, ns, mode, variant=0, splines=None, n_inner=None, knot_dim=True, col_of=None):
        assert mode in MODES and 0 <= ns and not (mode == "dens" and ns == 0)
        self.ns, self.mode, self.density = ns, mode, mode == "dens"
        self.name = f"ns{ns}-{mode}"
        terms, groups, cuts = [], [], []
        self.blocks = []  # (slot, size, kind) for drawing Lambda
        P = 0
        counts = splines or (SMALL_SPLINES if mode in ("lin0", "lin1", "lin2", "lin3") else LARGE_SPLINES)
        for d in range(ns):
            col = f"c{col_of[d] if col_of else d}"
            logx = (d + variant) % 2 == 0
            dens = self.density and d == 0
            grouped = d == 0 or (d == 2 and ns > 4)
            outside = S.OUTSIDE_ZERO if (d + variant) % 3 == 1 and not dens and not grouped else S.OUTSIDE_DROP
            lo, hi = (1.3, 9.6) if outside == S.OUTSIDE_ZERO else (1.05, 9.9)
            xi = (float(np.log(lo)), float(np.log(hi))) if logx else (lo, hi)
            n, knots, order = counts[(d + variant) % len(counts)], None, 4
            if knot_dim and ns >= 2 and d == ns - 1:  # explicit non-uniform knots: degree 0..3, a repeated interior knot
                degree = (variant + ns) % 4
                inner = n_inner or 6 + (variant + ns) % 5
                knots, n = explicit_knots(xi[0], xi[1], degree, inner)
                order = degree + 1
            t = S.Term(S.TERM_SPLINE_LINEAR if dens else S.TERM_SPLINE, [col], slots=[P], n_splines=n, logx=logx, outside=outside, xrange=(lo, hi),
                       knots=knots, order=order, name=f"spline[{col}]")
            t.xi_range = xi
            if grouped:
                grid = np.linspace(lo, hi, 150)
                gxi = np.clip(np.log(grid) if logx else grid, *xi)
                t.norm_group, t.grid_xi = len(groups), gxi
                groups.append(S.NormGroup(np.log(S.trapezoid_weights(grid)), name=f"Z[{col}]"))
            terms.append(t)
            self.blocks.append((P, n, "density" if dens else "spline"))
            P += n
        lin = {"lin0": 0, "lin1": 1, "lin2": 2, "lin3": 3, "param": 1, "dens": 1}[mode]
        for c, feat, off in [("c0", S.FEAT_LOG, -1.0), ("c1", S.FEAT_LOG1P, 0.5), ("c2", S.FEAT_NEG_LOG, 0.0)][:lin]:
            terms.append(S.Term(S.TERM_LINEAR, [c], slots=[P], cst=[off], feature=feat, name=f"lin[{c}]"))
            self.blocks.append((P, 1, "linear"))
            P += 1
        if mode == "param":  # the plan runs a power law as a linear term in log x and a per-evaluation normaliser
            terms.append(S.Term(S.TERM_TRUNCNORM, ["c3"], slots=[P, P + 1], cst=[1.0, 10.0], name="truncnorm[c3]"))
            terms.append(S.Term(S.TERM_POWERLAW, ["c4"], slots=[P + 2], cst=[1.0, 10.0], name="powerlaw[c4]"))
            self.blocks += [(P, 2, "truncnorm"), (P + 2, 1, "powerlaw")]
            P += 3
        terms.append(S.Term(S.TERM_STATIC, ["prior"], feature=S.FEAT_NEG_LOG, name="1/prior"))
        if variant % 2 == 0:
            cuts.append(S.Cut(S.CUT_RANGE, ["c7"], 1.1, 9.8))
        self.n_linear = lin + (mode == "param")
        self.n_param_terms = int(mode == "param")
        self.spec = S.ModelSpec(terms, groups, cuts, P)

    def draw_lambda(self, scale, seed):
        rng = np.random.default_rng(seed)
        lam = np.zeros(self.spec.n_params)
        for s, n, kind in self.blocks:
            if kind == "spline":
                lam[s : s + n] = scale * rng.standard_normal(n)
            elif kind == "density":  # a density must stay positive
                lam[s : s + n] = np.exp(scale * rng.standard_normal(n))
            elif kind == "linear":
                lam[s] = 0.5 * rng.standard_normal()
            elif kind == "truncnorm":
                lam[s : s + 2] = (5.0 + 0.5 * rng.standard_normal(), 1.5 + 0.2 * abs(rng.standard_normal()))
            else:
                lam[s] = -1.7 + 0.3 * rng.standard_normal()
        return lam


# ---- oracle ---------------------------------------------------------------------------------------------------------
def oracle(spec, pe_cols, inj_cols, lam):
    """popmodel.evaluate on a ragged catalog: the events of each size as one rectangular block (the injections once)."""
    first = spec.terms[0].cols[0]
    sizes = np.array([len(x) for x in pe_cols[first]])
    E, P = sizes.size, spec.n_params
    out = dict(logBF=np.empty(E), logNeff=np.empty(E), var=np.empty(E), J_logBF=np.empty((E, P)), J_logNeff=np.empty((E, P)))
    for b, s in enumerate(np.unique(sizes)):
        idx = np.flatnonzero(sizes == s)
        block = {k: np.stack([v[i] for i in idx]) for k, v in pe_cols.items()}
        ev = popmodel.evaluate(spec, block, inj_cols if b == 0 else {k: v[:1] for k, v in inj_cols.items()}, TOTAL_INJ, lam)
        for k in ("logBF", "logNeff", "var", "J_logBF", "J_logNeff"):
            out[k][idx] = ev[k]
        if b == 0:
            out.update({k: ev[k] for k in ("log_mu", "logNeff_inj", "var_inj", "J_log_mu", "J_logNeff_inj")})
    return out


def val_err(a, b):
    a, b = np.asarray(a, dtype=float), np.asarray(b, dtype=float)
    assert np.all(np.isfinite(a)) and np.all(np.isfinite(b))
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1.0)))


def grad_err(a, b):
    a, b = np.asarray(a, dtype=float), np.asarray(b, dtype=float)
    scale = np.maximum(np.abs(b), 1e-3 * np.max(np.abs(b)) + 1e-300)
    return float(np.max(np.abs(a - b) / scale))


# ---- geometries -----------------------------------------------------------------------------------------------------
def geometries(m, full):
    """(cta requested, n_deep, need_neff_grad) for one model.  Full: every geometry the model admits plus the requests
    the plan must lower (the CTA kernel with the N_eff moments, with no deep dim, or with a generic term).  Otherwise a
    subset that still runs every NS through each kernel with and without the N_eff moments."""
    top = min(m.ns, MAX_DEEP)
    cta_ok = m.ns >= 1 and m.mode in ("lin0", "lin1", "lin2")
    if full:
        out = [(False, nd, g2) for nd in range(top + 1) for g2 in (False, True)]
        if cta_ok:
            out += [(True, nd, False) for nd in range(1, top + 1)] + [(True, top, True), (True, 0, False)]
        elif m.ns >= 1:
            out += [(True, top, False)]
        return out
    out = [(False, m.ns % (top + 1), False), (False, (m.ns + 1) % (top + 1), True)]
    if cta_ok:
        out += [(True, max(1, top - m.ns % 2), False)]
    return out


def subset_models():
    """Per NS one model of each kernel family: register-resident linear terms (the CTA kernel's models) and the
    generic loop."""
    return [(ns, ("lin2", "lin0", "lin1")[ns % 3] if ns else "lin2") for ns in range(MAX_SPLINE_DIMS + 1)] + [
        (ns, ("lin3", "param", "dens")[ns % 3]) for ns in range(1, MAX_SPLINE_DIMS + 1)
    ] + [(0, "param")]


def all_models():
    return [(ns, mode) for ns in range(MAX_SPLINE_DIMS + 1) for mode in MODES if not (ns == 0 and mode in ("lin0", "dens"))]


def model_for(ns, mode):
    # the 6-dim models carry the 61-piece knot vector (the largest the library accepts)
    return Model(ns, mode, variant=ns + MODES.index(mode), n_inner=61 if ns == 6 else None)


@pytest.fixture(scope="module")
def matrix_full():
    return True


@pytest.fixture(scope="module")
def matrix_log():
    """What the matrix ran in this module: instantiation keys, lowered requests and the worst errors per kernel."""
    return dict(keys=set(), models=set(), lowered=[], worst={}, geometries=0)


def _note(log, kernel, what, err):
    w = log["worst"].setdefault(kernel, {"value": 0.0, "gradient": 0.0})
    w[what] = max(w[what], err)


def check_model(m, geometries_, monkeypatch, log, seed, cat_seed=None):
    """Run ``m`` through each geometry and check it against the oracle; returns the instantiation keys that ran."""
    pe_cols, inj_cols = catalog_columns(seed if cat_seed is None else cat_seed)
    E = len(pe_cols["c0"])
    lam, lam_b, lam_w = m.draw_lambda(0.3, seed), m.draw_lambda(0.3, seed + 1), m.draw_lambda(3.0, seed + 2)
    ref = {k: oracle(m.spec, pe_cols, inj_cols, x) for k, x in (("tight", lam), ("b", lam_b), ("wide", lam_w))}
    cat = capi.Catalog(pe_cols, inj_cols, TOTAL_INJ)
    rng = np.random.default_rng(seed)
    ran = set()
    try:
        for gi, (cta, nd, g2) in enumerate(geometries_):
            cs = int(rng.choice(CHUNK_STEPS))
            dev = gi % 2
            monkeypatch.setenv("GWI_CTA_KERNEL", str(int(cta)))
            monkeypatch.setenv("GWI_PLAN_DEVICE", str(dev))
            what = f"{m.name}: kernel={'cta' if cta else 'one-role'} n_deep={nd} g2={g2} chunk_steps={cs} plan_device={dev}"
            mdl = capi.Model(cat, m.spec, need_neff_grad=g2, chunk_steps=cs, n_deep=nd)
            try:
                ran |= _check_geometry(mdl, m, what, cta, nd, g2, dev, E, lam, lam_b, lam_w, ref, log)
            finally:
                mdl.close()
    finally:
        cat.close()
    log["keys"] |= ran
    return ran


def _check_geometry(mdl, m, what, cta, nd, g2, dev, E, lam, lam_b, lam_w, ref, log):
    info, plan0 = mdl.info(), mdl.read_plan(0)
    assert info["n_spline_dims"] == m.ns, what
    assert info["n_linear"] == m.n_linear and info["n_param_terms"] == m.n_param_terms, what
    assert info["plan_on_device"] == dev, what
    key = instantiation_key(info, plan0, g2, m.density)
    kernel = key[0]
    # the plan may lower a request: fewer deep dims for the shared-memory budget, the one-role kernel where the CTA
    # kernel does not apply (N_eff moments, a generic term, no deep dim); it never raises one
    assert info["n_deep"] <= nd, what
    if kernel == "cta":
        assert cta and not g2 and m.mode in ("lin0", "lin1", "lin2") and info["n_deep"] >= 1, what
    if info["n_deep"] != nd or (kernel == "cta") != cta:
        log["lowered"].append(dict(request=what, ran=list(key), block_threads=info["block_threads"]))
    log["geometries"] += 1
    ran = {key}

    # values and Jacobians
    for tag, x, vt, gt in (("tight", lam, VAL_RTOL, GRAD_RTOL), ("wide", lam_w, WIDE_VAL_RTOL, WIDE_GRAD_RTOL)):
        r, ev = mdl.evaluate(x), ref[tag]
        for k in ("logBF", "logNeff", "log_mu", "logNeff_inj"):
            e = val_err(r[k], ev[k])
            _note(log, kernel, "value", e)
            assert e <= vt, (what, tag, k, e)
        for k in ["J_logBF", "J_log_mu"] + (["J_logNeff", "J_logNeff_inj"] if g2 else []):
            e = grad_err(r[k], ev[k])
            _note(log, kernel, "gradient", e)
            assert e <= gt, (what, tag, k, e)

    # the likelihood and its gradient, with the a-priori / learned shift and with the exact maximum first
    def like(ev):
        return popmodel.hierarchical_log_likelihood(ev, E, marginalize_selection=g2, min_neff_cut=False)

    l_o, g_o, _ = like(ref["tight"])
    for exact in (False, True):
        mdl.set_exact_shift(exact)
        head, grad = mdl.loglike_host(lam, E, marginalize_selection=g2, min_neff_cut=False)
        assert head["passed"] == 1.0 and head["status"] == 0.0, (what, exact)
        e, eg = abs(head["log_l"] - l_o) / abs(l_o), float(np.max(np.abs(grad - g_o)) / np.max(np.abs(g_o)))
        _note(log, kernel, "value", e)
        _note(log, kernel, "gradient", eg)
        assert e <= VAL_RTOL and eg <= GRAD_RTOL, (what, "exact shift" if exact else "loglike", e, eg)
    mdl.set_exact_shift(False)
    ran.add(("ctamax",) if kernel == "cta" else ("max", m.ns))

    # three chains at different Lambda, each against its own oracle value
    ll, gg, head = mdl.loglike_batch(np.stack([lam, lam_b, lam_w]), E, marginalize_selection=g2, min_neff_cut=False)
    for c, (tag, vt, gt) in enumerate((("tight", VAL_RTOL, GRAD_RTOL), ("b", VAL_RTOL, GRAD_RTOL), ("wide", WIDE_VAL_RTOL, WIDE_GRAD_RTOL))):
        l_c, g_c, _ = like(ref[tag])
        assert head[c, 1] == 1.0, (what, "chain", c)
        e, eg = abs(ll[c] - l_c) / abs(l_c), float(np.max(np.abs(gg[c] - g_c)) / np.max(np.abs(g_c)))
        _note(log, kernel, "value", e)
        _note(log, kernel, "gradient", eg)
        assert e <= vt and eg <= gt, (what, "chain", c, e, eg)
    return ran


# ---- 1. the matrix --------------------------------------------------------------------------------------------------
def run_matrix_model(ns, mode, full, log, monkeypatch):
    m = model_for(ns, mode)
    check_model(m, geometries(m, full), monkeypatch, log, seed=1000 + 10 * ns + MODES.index(mode))
    log["models"].add((ns, mode))


@pytest.mark.parametrize("ns,mode", all_models())
def test_kernel_matrix(ns, mode, matrix_full, matrix_log, monkeypatch):
    run_matrix_model(ns, mode, matrix_full, matrix_log, monkeypatch)


# ---- 2. coverage ----------------------------------------------------------------------------------------------------
def test_every_reachable_instantiation_ran(matrix_full, matrix_log, monkeypatch):
    """Every key of the pick tables ran at least once, or is listed as unreachable with its reason: a new
    instantiation without a model that selects it fails here.  (Under the emulator's default subset: every NS through
    each kernel, with and without the N_eff moments.)  Models of the matrix that did not run in this session (a
    selection with -k) run here first."""
    for ns, mode in all_models() if matrix_full else subset_models():
        if (ns, mode) not in matrix_log["models"]:
            run_matrix_model(ns, mode, matrix_full, matrix_log, monkeypatch)
    ran = matrix_log["keys"]
    tables = one_role_keys() | cta_keys() | max_keys()
    assert len(one_role_keys()) == 280 and len(cta_keys()) == 78
    assert set(UNREACHABLE) <= tables and not (set(UNREACHABLE) & ran)
    assert ran <= tables, sorted(map(str, ran - tables))
    report = os.environ.get("GWI_KERNEL_MATRIX_REPORT")
    if report:
        with open(report, "w") as f:
            json.dump(dict(keys=sorted(map(list, ran), key=str), lowered=matrix_log["lowered"], worst=matrix_log["worst"], geometries=matrix_log["geometries"]), f, indent=1, default=str)
    print(f"kernel matrix: {matrix_log['geometries']} geometries, {len(ran)} instantiation keys; worst errors {matrix_log['worst']}")
    for low in matrix_log["lowered"]:
        print("lowered:", low)
    if matrix_full:
        missing = tables - ran - set(UNREACHABLE)
        assert not missing, sorted(map(str, missing))
    else:
        want = {("one", ns, g2) for ns in range(MAX_SPLINE_DIMS + 1) for g2 in (False, True)} | {("cta", ns) for ns in range(1, MAX_SPLINE_DIMS + 1)}
        got = {(k[0], k[1], k[4]) if k[0] == "one" else k[:2] for k in ran if k[0] in ("one", "cta")}
        assert want <= got, sorted(map(str, want - got))
        assert {("max", ns) for ns in range(MAX_SPLINE_DIMS + 1)} | {("ctamax",)} <= ran


# ---- 3. limits and edge geometries ----------------------------------------------------------------------------------
def _create(spec, **kw):
    pe_cols, inj_cols = catalog_columns(5, sizes=(3, 5), n_inj=200)
    cat = capi.Catalog(pe_cols, inj_cols, TOTAL_INJ)
    try:
        capi.Model(cat, spec, **kw).close()
    finally:
        cat.close()


def test_spline_dim_limit(monkeypatch, matrix_log):
    m = Model(MAX_SPLINE_DIMS, "lin1", variant=1)
    check_model(m, [(False, 2, False), (True, 2, False)], monkeypatch, matrix_log, seed=2001)
    over = Model(MAX_SPLINE_DIMS + 1, "lin1", variant=1, col_of=list(range(MAX_SPLINE_DIMS)) + [0])
    with pytest.raises(capi.GwiError, match="too many spline dimensions"):
        _create(over.spec)


def test_default_knot_spline_limit(monkeypatch, matrix_log):
    """At most 64 splines with the default knots (62 rows, J = 61 in the packed word); 65 are refused."""
    m = Model(3, "lin1", splines=(64, 5, 9))
    assert [t.n_splines for t in m.spec.terms[:2]] == [64, 5] and m.spec.terms[0].knots is None
    check_model(m, [(False, 1, False), (False, 0, True), (True, 1, False)], monkeypatch, matrix_log, seed=2002)
    over = Model(3, "lin1", splines=(65, 5, 9))
    with pytest.raises(capi.GwiError, match="bad spline description"):
        _create(over.spec)


def test_knot_piece_limit(monkeypatch, matrix_log):
    """An explicit knot vector may have 61 polynomial pieces inside its range; 62 are refused."""
    for degree in (3, 0):
        m = Model(2, "lin2", n_inner=61, variant=degree + 2)  # (variant + ns) % 4 == degree
        t = m.spec.terms[1]
        assert t.order == degree + 1 and knot_pieces(t.knots, *t.xi_range) == 61
        check_model(m, [(False, 2, False), (False, 1, True), (True, 1, False)], monkeypatch, matrix_log, seed=2003 + degree)
        over = Model(2, "lin2", n_inner=62, variant=degree + 2)
        t = over.spec.terms[1]
        assert knot_pieces(t.knots, *t.xi_range) == 62
        with pytest.raises(capi.GwiError, match="more than 61 polynomial pieces"):
            _create(over.spec)


@pytest.mark.parametrize("g2", [False, True])
def test_shared_memory_pressure(g2, monkeypatch, matrix_log):
    """8 dims x 64 splines: the shared-memory accumulators force fewer warps per block (and fewer deep dims); the
    model must still be created with the geometry the plan chose, and agree with the oracle."""
    m = Model(MAX_SPLINE_DIMS, "lin1", splines=(64,) * MAX_SPLINE_DIMS, knot_dim=False, variant=1)
    assert all(t.n_splines == 64 and t.knots is None for t in m.spec.terms[:MAX_SPLINE_DIMS])
    requests = [(False, MAX_DEEP, g2), (False, -1, g2), (True, 1, g2)]
    pe_cols, inj_cols = catalog_columns(7)
    cat = capi.Catalog(pe_cols, inj_cols, TOTAL_INJ)
    for cta, nd, _ in requests:
        monkeypatch.setenv("GWI_CTA_KERNEL", str(int(cta)))
        mdl = capi.Model(cat, m.spec, need_neff_grad=g2, n_deep=nd)
        info = mdl.info()
        mdl.close()
        print(f"8 x 64 splines, g2={g2}, cta requested={cta}, n_deep requested={nd}: n_deep={info['n_deep']} block_threads={info['block_threads']}"
              f" cta={bool(info['active_switches'] & 4)}")
        assert info["block_threads"] < 256
    cat.close()
    check_model(m, [(c, max(nd, 0), g) for c, nd, g in requests if nd >= 0], monkeypatch, matrix_log, seed=2010 + g2, cat_seed=7)


def test_device_builder_falls_back_to_the_host_builder(monkeypatch):
    """8 spline dims (48 key bits) and 65 536 events need 17 segment bits: more than the device builder's 64-bit sort
    key holds, so it hands the plan to the host builder.  The model must say so and agree with the oracle."""
    m = Model(MAX_SPLINE_DIMS, "lin1", variant=1)
    E = 65536
    rng = np.random.default_rng(11)
    sizes = 1 + (rng.random(E) < 0.5)
    pe_cols, inj_cols = catalog_columns(12, sizes=tuple(int(s) for s in sizes), n_inj=4000)
    lam = m.draw_lambda(0.3, 13)
    monkeypatch.setenv("GWI_PLAN_DEVICE", "1")
    cat = capi.Catalog(pe_cols, inj_cols, TOTAL_INJ)
    mdl = capi.Model(cat, m.spec, n_deep=2)
    try:
        assert mdl.info()["plan_on_device"] == 0
        r = mdl.evaluate(lam)
    finally:
        mdl.close()
        cat.close()
    # every event against the oracle's per-sample log-weights; the first 64 events and the injections with Jacobians
    x, valid, _ = popmodel.log_weights(m.spec, {k: np.concatenate(v) for k, v in pe_cols.items()}, lam)
    logZ = np.sum(popmodel.log_normalisers(m.spec, lam)[0])
    off = np.concatenate([[0], np.cumsum(sizes)])
    xm = np.maximum.reduceat(x, off[:-1])
    logBF = xm + np.log(np.add.reduceat(np.exp(x - np.repeat(xm, sizes)), off[:-1])) - np.log(sizes) - logZ
    assert val_err(r["logBF"], logBF) <= VAL_RTOL
    ev = oracle(m.spec, {k: v[:64] for k, v in pe_cols.items()}, inj_cols, lam)
    for k in ("log_mu", "logNeff_inj"):
        assert val_err(r[k], ev[k]) <= VAL_RTOL, k
    assert val_err(r["logNeff"][:64], ev["logNeff"]) <= VAL_RTOL
    assert grad_err(r["J_logBF"][:64], ev["J_logBF"]) <= GRAD_RTOL and grad_err(r["J_log_mu"], ev["J_log_mu"]) <= GRAD_RTOL
