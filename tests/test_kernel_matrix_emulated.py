"""CPU (no GPU): tests/test_kernel_matrix.py on the host warp emulator (tests/emu), without its `gpu` mark.

By default a deterministic subset of the matrix runs: every number of spline dims through each stream kernel, with and
without the N_eff moments, the max-only passes, the generic-term variant, and the limit and shared-memory tests.
GWI_KERNEL_MATRIX=full runs every model through every geometry, as on the GPU.  The device plan builder's fallback
test stays GPU-only: one evaluation of its 65 536 events takes about a minute here.
"""

import os

import pytest

from tests import emu
from tests import test_kernel_matrix as G

FULL = os.environ.get("GWI_KERNEL_MATRIX", "") == "full"
matrix_log = G.matrix_log


@pytest.fixture(scope="module")
def matrix_full():
    return FULL


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


@pytest.mark.parametrize("ns,mode", G.all_models() if FULL else G.subset_models())
def test_kernel_matrix(ns, mode, matrix_full, matrix_log, monkeypatch):
    G.run_matrix_model(ns, mode, matrix_full, matrix_log, monkeypatch)


# in this order: the coverage test reads what the matrix ran
test_every_reachable_instantiation_ran = G.test_every_reachable_instantiation_ran
test_spline_dim_limit = G.test_spline_dim_limit
test_default_knot_spline_limit = G.test_default_knot_spline_limit
test_knot_piece_limit = G.test_knot_piece_limit
test_shared_memory_pressure = G.test_shared_memory_pressure
