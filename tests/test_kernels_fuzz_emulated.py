"""CPU: randomised differential test of the kernel sources (on the host warp emulator, tests/emu) against
the NumPy oracle: random catalog sizes (down to one sample per event), spline counts, coefficient
scales, deep-dim splits, chunk lengths, N_eff gradients on / off and both epilogues.  Values to 1e-10,
Jacobians to 1e-8 (observed over 450 configurations: 1.4e-14 / 8.5e-14).  GWI_EMU_VARIANT selects a
variant build (e.g. ASan), GWI_FUZZ_CASES / GWI_FUZZ_SEED widen the search."""

import os

import numpy as np
import pytest

from gwinferno_b200 import capi, lowering, synthetic
from gwinferno_b200 import models as M
from gwinferno_b200.likelihood import PopulationLikelihood
from oracle import popmodel
from tests import emu


@pytest.fixture(scope="module", autouse=True)
def _emulated_device():
    variant = os.environ.get("GWI_EMU_VARIANT", "")
    try:
        if not variant:
            emu.build()
    except Exception as e:
        pytest.skip(f"host emulator build failed: {e}")
    emu.activate(variant)
    yield
    emu.deactivate()


def _rel(a, b):
    a, b = np.atleast_1d(np.asarray(a, float)), np.atleast_1d(np.asarray(b, float))
    # an event whose only sample has zero weight: log BF = -inf and log N_eff = nan in the reference, here too
    same = (np.isnan(a) & np.isnan(b)) | (np.isinf(a) & (a == b))
    if np.all(same):
        return 0.0
    assert np.all(np.isfinite(a[~same])) and np.all(np.isfinite(b[~same]))
    return float(np.max(np.abs(a[~same] - b[~same]) / np.maximum(np.abs(b[~same]), 1.0)))


def _grel(a, b):
    a, b = np.asarray(a, float), np.asarray(b, float)
    if np.max(np.abs(b)) < 1e-12:  # identically zero reference (d log N_eff of single-sample events)
        return float(np.max(np.abs(a - b)))
    return float(np.max(np.abs(a - b)) / np.max(np.abs(b)))


def test_random_configurations_against_the_oracle(monkeypatch):
    rng = np.random.default_rng(int(os.environ.get("GWI_FUZZ_SEED", "0")))
    n_cases = int(os.environ.get("GWI_FUZZ_CASES", "40"))
    done = 0
    for case in range(n_cases):
        E = int(rng.integers(1, 9))
        S = int(rng.choice([1, 3, 17, 64, 200, 333]))
        I = int(rng.choice([40, 500, 3000, 12000]))
        ns = dict(m1=int(rng.integers(5, 30)), q=int(rng.integers(5, 20)), a=int(rng.integers(5, 12)), t=int(rng.integers(5, 12)), z=int(rng.integers(5, 14)))
        pe, inj, const = synthetic.make_catalog(E, S, I, cfg=300 + case)
        mm = M.BSplinePrimaryBSplineRatio(ns["m1"], ns["q"], pe["mass_1"], inj["mass_1"], pe["mass_ratio"], inj["mass_ratio"], m1min=3.0, m2min=3.0, mmax=100.0,
                                          kwargs_m={"basis": M.LogXLogYBSpline}, kwargs_q={"basis": M.LogYBSpline})
        ma = M.BSplineIndependentSpinMagnitudes(ns["a"], ns["a"], pe["a_1"], pe["a_2"], inj["a_1"], inj["a_2"], normalize=True)
        mt = M.BSplineIndependentSpinTilts(ns["t"], ns["t"], pe["cos_tilt_1"], pe["cos_tilt_2"], inj["cos_tilt_1"], inj["cos_tilt_2"], normalize=True)
        mz = M.PowerlawSplineRedshiftModel(ns["z"], pe["redshift"], inj["redshift"])
        sc = float(rng.choice([0.1, 0.5, 2.0]))
        p = dict(m=sc * rng.standard_normal(ns["m1"]), q=sc * rng.standard_normal(ns["q"]), a1=sc * rng.standard_normal(ns["a"]), a2=sc * rng.standard_normal(ns["a"]),
                 t1=sc * rng.standard_normal(ns["t"]), t2=sc * rng.standard_normal(ns["t"]), lamb=np.float64(rng.uniform(-1, 4)), z=sc * rng.standard_normal(ns["z"]))

        def weights(d, pe_samples):
            w = mm(p["m"], p["q"], pe_samples=pe_samples) * ma(p["a1"], p["a2"], pe_samples=pe_samples) * mt(p["t1"], p["t2"], pe_samples=pe_samples)
            return w * mz(d["redshift"], p["lamb"], p["z"]) / d["prior"]

        pe_w, inj_w = weights(pe, True), weights(inj, False)
        low = lowering.lower(pe_w, inj_w)
        lam = lowering.flatten_params(pe_w, low.spec.n_params)
        g2 = bool(rng.integers(0, 2))
        nd = int(rng.choice([-1, 0, 1, 2, 3, 4]))
        cs = int(rng.choice([0, 2, 4, 8, 32, 128]))
        monkeypatch.setenv("GWI_CTA_KERNEL", str(int(rng.integers(0, 2))))  # both stream kernels (spline models qualify for the CTA-cooperative one)
        monkeypatch.setenv("GWI_PLAN_DEVICE", str(case % 2))  # both plan builders (host: plan.cpp, device kernels: plan_device.cu)
        try:
            eng = PopulationLikelihood(low, const["total_inj"], need_neff_grad=g2, chunk_steps=cs, n_deep=nd)
        except capi.GwiError as e:
            assert "bad spline description" in str(e)  # a one-sample catalog has a degenerate redshift range
            continue
        r = eng.evaluate(lam)
        eng.model.close()
        ev = popmodel.evaluate(low.spec, low.pe_cols, low.inj_cols, const["total_inj"], lam)
        what = f"case {case}: E={E} S={S} I={I} {ns} g2={g2} n_deep={nd} chunk_steps={cs} scale={sc}"
        for k in ("logBF", "logNeff", "log_mu", "logNeff_inj"):
            assert _rel(r[k], ev[k]) <= 1e-10, (what, k)
        for k in ["J_logBF", "J_log_mu"] + (["J_logNeff", "J_logNeff_inj"] if g2 else []):
            assert _grel(r[k], ev[k]) <= 1e-8, (what, k)
        done += 1
    assert done >= n_cases * 3 // 4


def test_random_model_families_against_the_oracle(monkeypatch):
    """The same for the three model families of BASELINE.json's configs (PL+Peak / Beta / iso+aligned with
    the generic-term kernel and its exact-max first pass; IID spins + IID masses; the full B-spline
    model) at random parameter points (360 configurations run by hand: worst 1.1e-14 / 4.0e-14)."""
    from gwinferno_b200 import workloads

    rng = np.random.default_rng(int(os.environ.get("GWI_FUZZ_SEED", "0")) + 1)
    for case in range(int(os.environ.get("GWI_FUZZ_CASES", "40")) // 2):
        fam = str(rng.choice(["plpeak", "bspline_iid", "bspline"]))
        E, S, I = int(rng.integers(1, 8)), int(rng.choice([2, 17, 100, 400])), int(rng.choice([200, 2000, 9000]))
        pe, inj, const = synthetic.make_catalog(E, S, I, cfg=500 + case)
        weights, params_fn = workloads.build_model(fam, pe, inj)
        low, lam, _ = workloads.lower_workload(weights, params_fn, pe, inj, seed=int(rng.integers(0, 1000)))
        g2, cs, nd = bool(rng.integers(0, 2)), int(rng.choice([0, 2, 8, 64])), int(rng.choice([-1, 0, 2, 4]))
        monkeypatch.setenv("GWI_CTA_KERNEL", str(int(rng.integers(0, 2))))  # both stream kernels (spline models qualify for the CTA-cooperative one)
        monkeypatch.setenv("GWI_PLAN_DEVICE", str(case % 2))  # both plan builders
        eng = PopulationLikelihood(low, const["total_inj"], need_neff_grad=g2, chunk_steps=cs, n_deep=nd)
        r = eng.evaluate(lam)
        eng.model.close()
        ev = popmodel.evaluate(low.spec, low.pe_cols, low.inj_cols, const["total_inj"], lam)
        what = f"case {case}: {fam} E={E} S={S} I={I} g2={g2} n_deep={nd} chunk_steps={cs}"
        for k in ("logBF", "logNeff", "log_mu", "logNeff_inj"):
            assert _rel(r[k], ev[k]) <= 1e-10, (what, k)
        for k in ["J_logBF", "J_log_mu"] + (["J_logNeff", "J_logNeff_inj"] if g2 else []):
            assert _grel(r[k], ev[k]) <= 1e-8, (what, k)
