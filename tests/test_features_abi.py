"""CPU-side checks of the feature ABI (include/rt_b200.h): the ctypes mirror of rt_denoise_features_params has the C
layout, and the library exports rt_render_features and rt_denoise_features and reports the version that introduced them."""
import ctypes as C
import os

import pytest


@pytest.fixture(scope="module")
def native():
    from ray_tracer_v1_b200 import _native
    if not os.path.exists(_native.LIB_PATH):
        _native.build()
    return _native


def test_denoise_features_params_layout_and_version(native):
    P = native.DenoiseFeaturesParams
    assert C.sizeof(P) == 24
    assert (P.radius.offset, P.patch_radius.offset, P.k.offset, P.k_f.offset, P.tau.offset, P.reserved_.offset) == \
        (0, 4, 8, 12, 16, 20)
    assert C.sizeof(native.DenoiseParams) == 16
    lib = native.load_symbols()
    assert lib.rt_version() >= 105
    for name in ("rt_render_features", "rt_denoise_features"):
        assert name in native.SIGNATURES and hasattr(lib, name)
