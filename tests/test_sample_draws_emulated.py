"""CPU (no GPU): tests/test_sample_draws.py on the host warp emulator (tests/emu), without its `gpu` mark.

The emulator runs a subset of the models and golden cases and fewer draws (test_sample_draws.emulated()); the full-size
cfg3 check is GPU only.
"""

import os

import pytest

from tests import emu
from tests import test_sample_draws as G


@pytest.fixture(scope="module", autouse=True)
def _emulated_device():
    variant = os.environ.get("GWI_EMU_VARIANT", "")
    try:
        if not variant:
            emu.build()
    except Exception as e:  # no g++ / not x86-64
        pytest.skip(f"host emulator build failed: {e}")
    emu.activate(variant)
    yield
    emu.deactivate()


test_sample_index_record = G.test_sample_index_record
test_host_plan_index_matches_model = G.test_host_plan_index_matches_model


@pytest.mark.parametrize("ns,mode", G.EMULATED_MODELS)
def test_log_weights_kernel_models(ns, mode, monkeypatch):
    G.check_log_weights(ns, mode, monkeypatch)


@pytest.mark.parametrize("name", G.EMULATED_CASES)
def test_log_weights_golden(name):
    G.check_golden(name)


test_draws_against_reference = G.test_draws_against_reference
test_draws_chi_square = G.test_draws_chi_square
test_isolation_from_the_likelihood = G.test_isolation_from_the_likelihood
test_dropin_posterior_predictive_plpeak = G.test_dropin_posterior_predictive_plpeak
