"""GPU (-m gpu): per-sample population log-weights and weighted draws (gwi_sample_log_weights / gwi_draw_samples).

A model created with keep_sample_index records, per padded stream position, the catalog position of its sample; the
log-weight pass scatters every sample's full log-weight to its catalog position and the draw pass samples each event (and
the injection set) with probability proportional to the weight, with counter-based uniforms (Philox4x32-10, counter
(k, s, 0, 0)).  Checked here, on the kernel-matrix catalogs and models (tests/test_kernel_matrix.py) and the golden
cases (tests/cases.py):

1. the index record: a permutation of the kept samples with -1 for padding, equal for both builders, and a plan that is
   otherwise bitwise the plan without it;
2. the log-weights against oracle/popmodel.py (|d| <= 1e-10 max(1, |x|), identical -inf sets) and against the model's
   own sums: logsumexp - log S_i is gwi_eval's logBF (1e-12 relative) and the golden logBF (1e-10);
3. independence of the plan geometry: bitwise across kernels, chunk lengths, deep dims and batch hints, 1e-13 across
   builders;
4. the draws: the NumPy reference below (cumsum + searchsorted on the same uniforms), zero-weight samples never drawn,
   -1 for an event without support, repeatable, and a chi-square test against the normalised weights;
5. isolation from the likelihood calls (results, speculative shift, graphs, last sites) and the argument checks;
6. the drop-in's posterior-predictive check on the parametric example's model;
7. the full cfg3 catalog (GPU only).

tests/test_sample_draws_emulated.py runs 1-6 on the host warp emulator (fewer models and draws).
"""

import ctypes as C

import numpy as np
import pytest
from scipy import special, stats

from gwinferno_b200 import capi, lowering
from gwinferno_b200.likelihood import PopulationLikelihood, hierarchical_likelihood
from gwinferno_b200.synthetic import philox4x32_10
from oracle import popmodel
from tests import cases
from tests import test_kernel_matrix as KM

pytestmark = pytest.mark.gpu

LOGW_TOL = 1e-10


def emulated():
    return hasattr(capi.load_library(), "gwi_emu_marker")


# ---- the NumPy reference of the draws ------------------------------------------------------------------------------
def uniforms(seed, s, k):
    """u01 of the first two words of Philox4x32-10 with counter (k, s, 0, 0), key (seed_lo, seed_hi)."""
    k = np.asarray(k, dtype=np.uint64)
    x, y, _, _ = philox4x32_10(k, np.full(k.shape, s, dtype=np.uint64), np.zeros(k.shape, np.uint64), np.zeros(k.shape, np.uint64), seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)
    return (((x << np.uint64(32)) | y) >> np.uint64(11)).astype(np.float64) * (1.0 / 9007199254740992.0)


def draw_indices(logw, offsets, seed, k_pe, k_inj):
    """Weighted draws from catalog-order log-weights: segment s (event s, the injections last) covers
    [offsets[s], offsets[s+1]).  Returns (pe[E, k_pe], inj[k_inj], near): near counts the draws whose r lies within
    1e-12 of the total of a prefix boundary (where rounding may pick the neighbour)."""
    E = len(offsets) - 2
    out, near = [], 0
    for s in range(E + 1):
        k = k_pe if s < E else k_inj
        x = logw[offsets[s] : offsets[s + 1]]
        m = np.max(x) if x.size else -np.inf
        if not np.isfinite(m):
            out.append(np.full(k, -1, dtype=np.int64))
            continue
        c = np.cumsum(np.exp(x - m))
        r = np.minimum(uniforms(seed, s, np.arange(k)) * c[-1], np.nextafter(c[-1], 0.0))
        idx = np.searchsorted(c, r, side="right")
        lo = np.where(idx > 0, c[np.maximum(idx - 1, 0)], 0.0)
        near += int(np.sum((np.abs(c[idx] - r) <= 1e-12 * c[-1]) | (np.abs(r - lo) <= 1e-12 * c[-1])))
        out.append(idx.astype(np.int64))
    return np.stack(out[:E]).reshape(E, k_pe) if E else np.zeros((0, k_pe), np.int64), out[E], near


# ---- helpers --------------------------------------------------------------------------------------------------------
def catalog(seed, n_inj=KM.N_INJ, empty_event=False):
    """A kernel-matrix catalog; empty_event appends an event of 5 samples outside every model's support."""
    pe, inj = KM.catalog_columns(seed, n_inj=n_inj)
    if empty_event:
        for k in pe:
            pe[k].append(np.full(5, 0.5) if k != "prior" else np.ones(5))
    return pe, inj


def seg_offsets(pe, inj):
    sizes = [len(x) for x in pe["c0"]]
    return np.concatenate([[0], np.cumsum(sizes), [sum(sizes) + len(inj["c0"])]]).astype(np.int64)


def oracle_logw(spec, pe, inj, lam):
    cols = {k: np.concatenate([np.concatenate(pe[k]), inj[k]]) for k in pe}
    x, valid, _ = popmodel.log_weights(spec, cols, lam)
    return x - np.sum(popmodel.log_normalisers(spec, lam)[0]), valid


def assert_logw(got, ref, what):
    fin = np.isfinite(ref)
    assert np.array_equal(np.isfinite(got), fin) and not np.any(np.isnan(got)), what
    assert np.all(got[~fin] == -np.inf), what
    err = np.max(np.abs(got[fin] - ref[fin]) / np.maximum(1.0, np.abs(ref[fin]))) if fin.any() else 0.0
    assert err <= LOGW_TOL, (what, err)


def logmeans(logw, off, n_total_inj):
    """logsumexp - log S per event, and log mu of the injections."""
    E = len(off) - 2
    ev = np.array([special.logsumexp(logw[off[i] : off[i + 1]]) - np.log(off[i + 1] - off[i]) for i in range(E)])
    return ev, special.logsumexp(logw[off[E] :]) - np.log(n_total_inj)


def rel(a, b):
    return float(np.max(np.abs(np.asarray(a) - np.asarray(b)) / np.maximum(np.abs(np.asarray(b)), 1e-300)))


def make(cat, spec, monkeypatch, cta=0, dev=0, **kw):
    monkeypatch.setenv("GWI_CTA_KERNEL", str(int(cta)))
    monkeypatch.setenv("GWI_PLAN_DEVICE", str(int(dev)))
    return capi.Model(cat, spec, **kw)


def index_models():
    return [(2, "lin1"), (3, "param"), (2, "dens")] if emulated() else [(2, "lin1"), (4, "lin2"), (3, "param"), (2, "dens"), (0, "param")]


ALL_MODELS = [(ns, mode) for ns in range(KM.MAX_SPLINE_DIMS + 1) for mode in KM.MODES if not (ns == 0 and mode in ("lin0", "dens"))]
EMULATED_MODELS = [(1, "lin2"), (2, "param"), (3, "dens"), (0, "param")]  # tests/test_sample_draws_emulated.py
EMULATED_CASES = ["bspline_full", "plpeak", "bspline_redshift_default", "bspline_knots_density"]


# ---- 1. the index record ----------------------------------------------------------------------------------------------
def test_sample_index_record(monkeypatch):
    for ns, mode in index_models():
        m = KM.model_for(ns, mode)
        pe, inj = catalog(100 + ns)
        cat = capi.Catalog(pe, inj, KM.TOTAL_INJ)
        _, valid = oracle_logw(m.spec, pe, inj, m.draw_lambda(0.3, 1))
        n_cat = valid.size
        try:
            for cta in (0, 1):
                for cs in (0, 2, 32):
                    idx = {}
                    for dev in (0, 1):
                        what = f"{m.name} cta={cta} chunk_steps={cs} plan_device={dev}"
                        a = make(cat, m.spec, monkeypatch, cta, dev, chunk_steps=cs, keep_sample_index=True)
                        b = make(cat, m.spec, monkeypatch, cta, dev, chunk_steps=cs)
                        try:
                            r = a.read_plan(7)
                            assert r.size == a.info()["n_padded"] and b.read_plan(7).size == 0, what
                            kept = r[r >= 0]
                            assert np.unique(kept).size == kept.size and np.all(kept < n_cat), what
                            assert np.all(r[r < 0] == -1), what
                            mask = np.zeros(n_cat, bool)
                            mask[kept] = True
                            # the plan drops what has no support; a parametric term or a spline density may still give a
                            # kept sample weight 0 (its log-weight is then -inf)
                            assert np.all(mask[valid]), what
                            if mode not in ("param", "dens"):
                                assert np.array_equal(mask, valid), what
                            for w in (1, 2, 3, 5, 6):
                                assert np.array_equal(a.read_plan(w), b.read_plan(w)), (what, w)
                            idx[dev] = r
                        finally:
                            a.close()
                            b.close()
                    assert np.array_equal(idx[0], idx[1]), (m.name, cta, cs)
        finally:
            cat.close()


def test_host_plan_index_matches_model(monkeypatch):
    m = KM.model_for(2, "lin2")
    pe, inj = catalog(7)
    cat = capi.Catalog(pe, inj, KM.TOTAL_INJ)
    try:
        hp = capi.HostPlan(cat, m.spec, keep_sample_index=True)
        mdl = make(cat, m.spec, monkeypatch, 0, 0, keep_sample_index=True)
        assert np.array_equal(hp.read(7), mdl.read_plan(7))
        assert capi.HostPlan(cat, m.spec).read(7).size == 0
        mdl.close()
        hp.close()
    finally:
        cat.close()


# ---- 2. + 3. log-weights against the oracle, the model's own sums, across geometries -------------------------------
def check_log_weights(ns, mode, monkeypatch):
    m = KM.model_for(ns, mode)
    pe, inj = catalog(300 + 10 * ns + KM.MODES.index(mode))
    off = seg_offsets(pe, inj)
    cat = capi.Catalog(pe, inj, KM.TOTAL_INJ)
    lam = m.draw_lambda(0.3, 5 + ns)
    ref, _ = oracle_logw(m.spec, pe, inj, lam)
    top = min(ns, KM.MAX_DEEP)
    geoms = [(0, 0, 0, 0), (0, top, 2, 0), (0, 0, 32, 4)]
    if ns >= 1 and mode in ("lin0", "lin1", "lin2"):
        geoms.append((1, max(1, top), 0, 0))
    if emulated():
        geoms = geoms[:2]
    base, base_draws = None, None
    try:
        for dev in (0, 1):
            for cta, nd, cs, bh in geoms:
                what = f"{m.name} cta={cta} n_deep={nd} chunk_steps={cs} batch_hint={bh} plan_device={dev}"
                mdl = make(cat, m.spec, monkeypatch, cta, dev, n_deep=nd, chunk_steps=cs, batch_hint=bh, keep_sample_index=True)
                try:
                    x = mdl.sample_log_weights(lam)
                    d = mdl.draw_samples(lam, 11, 3, 7)
                    if base is None:
                        assert_logw(x, ref, what)
                        r = mdl.evaluate(lam, jacobians=False)
                        ev, lmu = logmeans(x, off, KM.TOTAL_INJ)
                        assert rel(ev, r["logBF"]) <= 1e-12 and rel(lmu, r["log_mu"]) <= 1e-12, what
                        base, base_draws, base_dev = x, d, dev
                    elif dev == base_dev:
                        assert np.array_equal(x, base) and all(np.array_equal(a, b) for a, b in zip(d, base_draws)), what
                    else:
                        fin = np.isfinite(base)
                        assert np.array_equal(np.isfinite(x), fin) and rel(x[fin], base[fin]) <= 1e-13, what
                finally:
                    mdl.close()
    finally:
        cat.close()


@pytest.mark.parametrize("ns,mode", ALL_MODELS)
def test_log_weights_kernel_models(ns, mode, monkeypatch):
    check_log_weights(ns, mode, monkeypatch)


@pytest.mark.parametrize("name", cases.GOLDEN_CASES + cases.HOST_GLUE_CASES)
def test_log_weights_golden(name):
    check_golden(name)


def check_golden(name):
    c = cases.load_case(name)
    eng = PopulationLikelihood.from_weights(c.pe_w, c.inj_w, c.total_inj, keep_sample_index=True)
    try:
        logZ_host = lowering.host_log_norm(c.pe_w, eng.n_params)[0]
        pe, inj = eng.sample_log_weights(c.Lam, host_log_norm=logZ_host)
        E, S = c.low.pe_cols[next(iter(c.low.pe_cols))].shape
        ref_pe, _ = oracle_logw(c.low.spec, {k: list(v) for k, v in c.low.pe_cols.items()}, {k: v[:0] for k, v in c.low.inj_cols.items()}, c.Lam)
        ref_inj, _ = popmodel.log_weights(c.low.spec, c.low.inj_cols, c.Lam)[:2]
        ref_inj = ref_inj - np.sum(popmodel.log_normalisers(c.low.spec, c.Lam)[0])
        assert pe.shape == (E, S)
        assert_logw(pe.reshape(-1), ref_pe - logZ_host, name)
        assert_logw(inj, ref_inj - logZ_host, name)
        r = eng.evaluate(c.Lam, jacobians=False)
        ev = special.logsumexp(pe, axis=1) - np.log(S)
        lmu = special.logsumexp(inj) - np.log(c.total_inj)
        assert rel(ev, r["logBF"] - logZ_host) <= 1e-12 and rel(lmu, r["log_mu"] - logZ_host) <= 1e-12
        assert np.max(np.abs(ev - c.out["logBF"]) / np.maximum(1.0, np.abs(c.out["logBF"]))) <= 1e-10
        assert abs(lmu - float(c.out["log_mu"])) <= 1e-10 * max(1.0, abs(float(c.out["log_mu"])))
    finally:
        eng.model.close()
        eng.catalog.close()


# ---- 4. draws ---------------------------------------------------------------------------------------------------------
def test_draws_against_reference(monkeypatch):
    m = KM.model_for(2, "param")
    pe, inj = catalog(21, empty_event=True)
    off = seg_offsets(pe, inj)
    E = len(pe["c0"])
    cat = capi.Catalog(pe, inj, KM.TOTAL_INJ)
    lam = m.draw_lambda(0.3, 3)
    try:
        mdl = make(cat, m.spec, monkeypatch, 0, 0, keep_sample_index=True)
        x = mdl.sample_log_weights(lam)
        k_pe, k_inj = (40, 300) if emulated() else (400, 5000)
        for seed in (0, 12345, 2**40 + 7):
            d_pe, d_inj = mdl.draw_samples(lam, seed, k_pe, k_inj)
            o_pe, o_inj, near = draw_indices(x, off, seed, k_pe, k_inj)
            assert near == 0, near  # expected: no uniform this close to a prefix boundary
            assert np.array_equal(d_pe, o_pe) and np.array_equal(d_inj, o_inj), seed
            assert np.all(d_pe[E - 1] == -1)  # the event outside every support
            for i in range(E - 1):
                assert np.all(np.isfinite(x[off[i] + d_pe[i]])), i  # zero-weight samples are never drawn
            assert np.all(np.isfinite(x[off[E] + d_inj]))
            again = mdl.draw_samples(lam, seed, k_pe, k_inj)
            assert np.array_equal(again[0], d_pe) and np.array_equal(again[1], d_inj)
        z_pe, z_inj = mdl.draw_samples(lam, 1, 0, 0)
        assert z_pe.shape == (E, 0) and z_inj.size == 0
        mdl.close()
    finally:
        cat.close()


def chi2_p(idx, logw):
    p = np.exp(logw - np.max(logw))
    p /= p.sum()
    counts = np.bincount(idx, minlength=p.size)
    assert np.all(counts[p == 0] == 0)
    expected = p * idx.size
    keep = expected > 0
    return stats.chisquare(counts[keep], expected[keep]).pvalue


def test_draws_chi_square(monkeypatch):
    """A 37-sample event and a 2000-injection set: the draw frequencies against the normalised weights."""
    m = KM.model_for(1, "lin2")
    pe, inj = catalog(31, n_inj=2000)
    off = seg_offsets(pe, inj)
    i37 = [len(v) for v in pe["c0"]].index(37)
    cat = capi.Catalog(pe, inj, KM.TOTAL_INJ)
    n = 20_000 if emulated() else 200_000
    try:
        mdl = make(cat, m.spec, monkeypatch, 0, 0, keep_sample_index=True)
        lam = m.draw_lambda(0.3, 9)
        x = mdl.sample_log_weights(lam)
        d_pe, d_inj = mdl.draw_samples(lam, 77, n, n)
        p_ev = chi2_p(d_pe[i37], x[off[i37] : off[i37 + 1]])
        p_inj = chi2_p(d_inj, x[off[-2] :])
        print(f"chi-square p-values: 37-sample event {p_ev:.3g}, 2000 injections {p_inj:.3g} ({n} draws each)")
        assert p_ev >= 1e-6 and p_inj >= 1e-6
        mdl.close()
    finally:
        cat.close()


# ---- 5. isolation and arguments --------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["lin2", "param"])  # graph-replayed host call / speculative shift
def test_isolation_from_the_likelihood(mode, monkeypatch):
    m = KM.model_for(2, mode)
    pe, inj = catalog(41)
    E = len(pe["c0"])
    cat = capi.Catalog(pe, inj, KM.TOTAL_INJ)
    lam, lam2 = m.draw_lambda(0.3, 1), m.draw_lambda(0.3, 2)
    try:
        plain = make(cat, m.spec, monkeypatch, 0, 0, keep_sample_index=True)
        mixed = make(cat, m.spec, monkeypatch, 0, 0, keep_sample_index=True)
        want = [plain.loglike_host(x, E, min_neff_cut=False) for x in (lam, lam2)]
        first = mixed.loglike_host(lam, E, min_neff_cut=False)
        sites = mixed.last_sites()
        mixed.sample_log_weights(lam2 * 1.1)
        mixed.draw_samples(lam2 * 0.9, 5, 2, 3)
        assert np.array_equal(mixed.last_sites(), sites)
        second = mixed.loglike_host(lam2, E, min_neff_cut=False)
        for (h0, g0), (h1, g1) in zip(want, (first, second)):
            assert h0 == h1 and np.array_equal(g0, g1)
        plain.close()
        mixed.close()
        # a model without the index, and bad arguments
        lib = capi.load_library()
        no = make(cat, m.spec, monkeypatch, 0, 0)
        with pytest.raises(capi.GwiError) as e:
            no.sample_log_weights(lam)
        assert e.value.code == -4
        assert lib.gwi_draw_samples(no.handle, C.c_void_p(8), 0, 1, 1, C.c_void_p(8), None) == -4
        no.close()
        mdl = make(cat, m.spec, monkeypatch, 0, 0, keep_sample_index=True)
        buf = capi.DeviceBuffer(16)
        assert lib.gwi_sample_log_weights(mdl.handle, None, C.c_void_p(buf.ptr), None) == -1
        assert lib.gwi_sample_log_weights(mdl.handle, C.c_void_p(buf.ptr), None, None) == -1
        assert lib.gwi_sample_log_weights(None, C.c_void_p(buf.ptr), C.c_void_p(buf.ptr), None) == -1
        assert lib.gwi_draw_samples(mdl.handle, C.c_void_p(buf.ptr), 0, -1, 1, C.c_void_p(buf.ptr), None) == -1
        assert lib.gwi_draw_samples(mdl.handle, C.c_void_p(buf.ptr), 0, 1, -1, C.c_void_p(buf.ptr), None) == -1
        assert lib.gwi_draw_samples(mdl.handle, C.c_void_p(buf.ptr), 0, 1, 1, None, None) == -1
        buf.free()
        mdl.close()
    finally:
        cat.close()


# ---- 6. the drop-in's posterior-predictive check ---------------------------------------------------------------------
def test_dropin_posterior_predictive_plpeak():
    c = cases.load_case("plpeak")
    names = ["mass_1", "mass_ratio", "redshift"]
    base = hierarchical_likelihood(c.pe_w, c.inj_w, c.total_inj, c.Nobs, c.Tobs, **c.like_kw)
    res = hierarchical_likelihood(c.pe_w, c.inj_w, c.total_inj, c.Nobs, c.Tobs, posterior_predictive_check=True, param_names=names, pedata=c.pe,
                                  injdata=c.inj, rngkey=3, **c.like_kw)
    assert res.log_likelihood == base.log_likelihood and np.array_equal(res.grad_flat, base.grad_flat)
    E = c.pe["mass_1"].shape[0]
    x, _ = oracle_logw(c.low.spec, {k: list(v) for k, v in c.low.pe_cols.items()}, c.low.inj_cols, c.Lam)
    off = np.concatenate([np.arange(E + 1) * c.pe["mass_1"].shape[1], [x.size]])
    o_pe, o_inj, near = draw_indices(x, off, 3, 1, E)
    assert near == 0
    assert np.array_equal(res.ppc["obs_index"], o_pe[:, 0]) and np.array_equal(res.ppc["pred_index"], o_inj)
    for n in names:
        for i in range(E):
            assert res.sites[f"{n}_obs_event_{i}"] == c.pe[n][i, o_pe[i, 0]]
            assert res.sites[f"{n}_pred_event_{i}"] == c.inj[n][o_inj[i]]
        assert np.array_equal(res.ppc["obs"][n], c.pe[n][np.arange(E), o_pe[:, 0]])
    with pytest.raises(NotImplementedError):
        hierarchical_likelihood(c.pe_w, c.inj_w, c.total_inj, c.Nobs, c.Tobs, posterior_predictive_check=True, pedata=c.pe, injdata=c.inj, **c.like_kw)


# ---- 7. full size (GPU only) ------------------------------------------------------------------------------------------
def test_cfg3_full_size():
    from gwinferno_b200 import workloads

    pe, inj, const, z_range = workloads.shard_catalog("cfg3", 0, 1, scale=1.0, all_reduce_minmax=lambda lo, hi: (lo, hi))
    weights, params_fn = workloads.build_model(const["family"], pe, inj, z_range=z_range)
    low, lam, _ = workloads.lower_workload(weights, params_fn, pe, inj)
    E = low.pe_cols[next(iter(low.pe_cols))].shape[0]
    with_idx = PopulationLikelihood(low, const["total_inj"], keep_sample_index=True)
    plain = PopulationLikelihood(low, const["total_inj"])
    try:
        for x in (lam, lowering.flatten_params(weights(pe, True, params_fn(5)), low.spec.n_params)):
            a, b = with_idx.loglike(x, Nobs=E), plain.loglike(x, Nobs=E)
            assert a[0] == b[0] and np.array_equal(a[1], b[1]) and a[2] == b[2]
        pe_w, inj_w = with_idx.sample_log_weights(lam)
        r = with_idx.evaluate(lam, jacobians=False)
        S = pe_w.shape[1]
        assert rel(special.logsumexp(pe_w, axis=1) - np.log(S), r["logBF"]) <= 1e-12
        assert rel(special.logsumexp(inj_w) - np.log(const["total_inj"]), r["log_mu"]) <= 1e-12
        d1 = with_idx.posterior_predictive(lam, seed=9)
        d2 = with_idx.posterior_predictive(lam, seed=9)
        assert np.array_equal(d1[0], d2[0]) and np.array_equal(d1[1], d2[1]) and np.all(d1[0] >= 0) and np.all(d1[1] >= 0)
    finally:
        for e in (with_idx, plain):
            e.model.close()
            e.catalog.close()
