"""CPU-side checks of the denoise ABI (include/rt_b200.h): the ctypes mirror of rt_denoise_params has the C layout, and
the library that exports rt_denoise reports the version that introduced it."""
import ctypes as C
import os

import pytest


@pytest.fixture(scope="module")
def native():
    from ray_tracer_v1_b200 import _native
    if not os.path.exists(_native.LIB_PATH):
        _native.build()
    return _native


def test_denoise_params_layout_and_version(native):
    P = native.DenoiseParams
    assert C.sizeof(P) == 16
    assert (P.radius.offset, P.patch_radius.offset, P.k.offset, P.reserved_.offset) == (0, 4, 8, 12)
    lib = native.load_symbols()
    assert lib.rt_version() >= 104
    assert "rt_denoise" in native.SIGNATURES and hasattr(lib, "rt_denoise")
