"""CPU (no GPU): the CUDA kernel SOURCES under the host warp emulator (tests/emu).

tests/emu compiles gwinferno_b200/csrc/{kernels.cu, stream.cuh, api.cu, plan.cpp} with g++ against a
stand-in <cuda_runtime.h> in which every CUDA thread is a fiber (warp shuffles / ballots / barriers
are real exchanges between the fibers of a warp, blocks run on OS threads).  The parity tests of
tests/test_gpu_parity.py are then run unchanged through the same C-ABI entry points: golden vectors
of the reference, the oracle on seeded catalogs, ragged / masked / empty inputs, shard combine,
chain batches.  This checks the kernels' index arithmetic, accumulator layouts, reductions and
likelihood glue in a container without a GPU; it says nothing about speed, and it is test
infrastructure only -- the product library has no CPU path and the binding refuses the emulator
build (test_product_binding_refuses_the_emulator_build).
"""

import os

import pytest

from gwinferno_b200 import capi
from tests import emu
from tests import test_gpu_parity as G

# fixtures and tests of the GPU module, collected here WITHOUT its `gpu` mark
golden = G.golden
medium = G.medium
cfg2 = G.cfg2
ppd_ref = G.ppd_ref
for _name in dir(G):
    if _name.startswith("test_"):
        globals()[_name] = getattr(G, _name)
del _name


@pytest.fixture(scope="module", autouse=True)
def _emulated_device():
    variant = os.environ.get("GWI_EMU_VARIANT", "")  # a variant build (tests/emu/Makefile VARIANT=, e.g. ASan), built by hand
    try:
        if not variant:
            emu.build()
    except Exception as e:  # no g++ / not x86-64
        pytest.skip(f"host emulator build failed: {e}")
    emu.activate(variant)
    yield
    emu.deactivate()


def test_product_binding_refuses_the_emulator_build():
    saved = (capi._lib, capi.LIB_PATH)
    try:
        capi._lib, capi.LIB_PATH = None, emu.library_path()
        with pytest.raises(capi.GwiError, match="host-emulator build"):
            capi.load_library()
    finally:
        capi._lib, capi.LIB_PATH = saved


def test_emulator_is_not_part_of_the_product_library():
    import ctypes

    prod = os.path.join(os.path.dirname(capi.__file__), "libgwi.so")
    if not os.path.exists(prod):
        pytest.skip("libgwi.so not built")
    assert not hasattr(ctypes.CDLL(prod), "gwi_emu_marker")
