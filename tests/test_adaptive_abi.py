"""CPU-side checks of the adaptive-frame ABI (include/rt_b200.h): the ctypes mirror of rt_adaptive_params has the C
layout, and the library that exports rt_render_path_adaptive reports the version that introduced it."""
import ctypes as C
import os

import pytest


@pytest.fixture(scope="module")
def native():
    from ray_tracer_v1_b200 import _native
    if not os.path.exists(_native.LIB_PATH):
        _native.build()
    return _native


def test_adaptive_params_layout_and_version(native):
    assert C.sizeof(native.AdaptiveParams) == 16
    assert native.AdaptiveParams.min_spp.offset == 0 and native.AdaptiveParams.tolerance.offset == 8
    lib = native.load_symbols()
    assert lib.rt_version() >= 103
    assert "rt_render_path_adaptive" in native.SIGNATURES and hasattr(lib, "rt_render_path_adaptive")
