"""CPU (no GPU): tests/test_param_terms_exact.py on the host warp emulator (tests/emu), without its `gpu` mark.

The emulator evaluates erf, erfc, expm1, lgamma and pow with the host's libm; the GPU run of the same tests is the one
that checks CUDA's.
"""

import os

import pytest

from tests import emu
from tests import test_param_terms_exact as G


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


test_term_points = G.test_term_points
test_term_batch = G.test_term_batch
