"""CPU: the kernel sources at the sizes BASELINE.json names, on the host warp emulator, against the
plain-C oracle (an independent implementation from the raw coordinates: no plan, no sorting).

The emulator runs the unmodified stream / reduce / finish / partial / combine kernels with the plan
geometry of a 148-SM device (GWI_EMU_SMS), so slices, chunks, guided tail, reduction-tree depth and the
sorted-run lengths are those of the real run at that size.  Default: config 5 at a quarter of its size
and config 3 at 5 % (seconds each).  GWI_TEST_FULL_SIZE=1 adds config 3 at FULL size (300 x 10 000 +
1e8 injections; ~25 GB of host memory, about two minutes) -- run by hand, result quoted in DESIGN.md.
"""

import os

import numpy as np
import pytest

from gwinferno_b200 import workloads
from gwinferno_b200.likelihood import PopulationLikelihood
from oracle import c_oracle, popmodel
from tests import emu


@pytest.fixture(scope="module", autouse=True)
def _emulated_b200():
    old = os.environ.get("GWI_EMU_SMS")
    os.environ["GWI_EMU_SMS"] = "148"
    variant = os.environ.get("GWI_EMU_VARIANT", "")  # a variant build made by hand (tests/emu/Makefile VARIANT=, e.g. ASan)
    try:
        if not variant:
            emu.build()
        c_oracle.build()
    except Exception as e:
        pytest.skip(f"build failed: {e}")
    emu.activate(variant)
    yield
    emu.deactivate()
    if old is None:
        os.environ.pop("GWI_EMU_SMS", None)
    else:
        os.environ["GWI_EMU_SMS"] = old


def _check(name, scale, world=1, min_neff_cut=True):
    pe, inj, const, z_range = workloads.shard_catalog(name, 0, world, scale=scale, all_reduce_minmax=lambda lo, hi: (lo, hi))
    weights, params_fn = workloads.build_model(const["family"], pe, inj, z_range=z_range)
    low, lam, _ = workloads.lower_workload(weights, params_fn, pe, inj)
    eng = PopulationLikelihood(low, const["total_inj"])
    info = eng.info()
    E = low.pe_cols[next(iter(low.pe_cols))].shape[0]
    log_l, grad, head = eng.loglike(lam, Nobs=E, min_neff_cut=min_neff_cut)
    eng.model.close()
    ev = c_oracle.evaluate(low.spec, low.pe_cols, low.inj_cols, const["total_inj"], lam, want_jac=True, want_neff_jac=False, n_threads=os.cpu_count() or 1)
    l_o, g_o, _ = popmodel.hierarchical_log_likelihood(ev, E, min_neff_cut=min_neff_cut)
    assert head["passed"] == 1.0 and head["status"] == 0.0
    assert abs(log_l - l_o) <= 1e-10 * abs(l_o)
    assert np.max(np.abs(grad - g_o)) <= 1e-8 * np.max(np.abs(g_o))
    return info, abs(log_l - l_o) / abs(l_o), np.max(np.abs(grad - g_o)) / np.max(np.abs(g_o))


def test_cfg5_quarter_size():
    info, el, eg = _check("cfg5", 0.25)
    assert info["n_padded"] > 5_000_000


def test_cfg3_five_percent():
    # scaled-down events have fewer samples than the N_eff cut asks for (N_eff,i > 300 events): compare without it
    info, el, eg = _check("cfg3", 0.05, min_neff_cut=False)
    assert info["n_padded"] > 5_000_000


def test_cfg3_rank0_of_8_at_ten_percent():
    _check("cfg3", 0.1, world=8, min_neff_cut=False)


@pytest.mark.skipif(os.environ.get("GWI_TEST_FULL_SIZE") != "1", reason="~25 GB of host memory, two minutes: set GWI_TEST_FULL_SIZE=1")
def test_cfg3_full_size():
    info, el, eg = _check("cfg3", 1.0)
    assert info["n_padded"] > 100_000_000
    print(f"cfg3 full size on the emulator vs the C oracle: rel err log L {el:.2e}, gradient {eg:.2e}, {info['n_chunks']} chunks")
