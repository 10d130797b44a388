"""CPU-side checks of the row-band filter ABI (include/rt_b200.h): the library exports rt_denoise_rows,
rt_denoise_features_rows and rt_denoise_halo, reports the version that introduced them, and rt_denoise_halo gives the
halo depth of each filter and rejects the parameters the filters reject."""
import os

import pytest


@pytest.fixture(scope="module")
def native():
    from ray_tracer_v1_b200 import _native
    if not os.path.exists(_native.LIB_PATH):
        _native.build()
    return _native


def test_rows_symbols_and_version(native):
    lib = native.load_symbols()
    assert lib.rt_version() >= 106
    for name in ("rt_denoise_rows", "rt_denoise_features_rows", "rt_denoise_halo"):
        assert name in native.SIGNATURES and hasattr(lib, name)


def test_denoise_halo(native):
    for r in range(16):
        for f in range(6):
            assert native.denoise_halo(r, f) == r + f
            assert native.denoise_halo(r, f, features=True) == max(r + f, 1)
    assert native.denoise_halo() == 13 and native.denoise_halo(features=True) == 13


def test_denoise_halo_rejections(native):
    import ctypes as C
    lib = native.load_symbols()
    h = C.c_int32(-7)
    for (r, f), msg in (((-1, 0), "radius"), ((16, 0), "radius"), ((0, -1), "patch_radius"), ((0, 6), "patch_radius")):
        assert lib.rt_denoise_halo(r, f, 0, C.byref(h)) == 1
        assert msg in lib.rt_last_error().decode()
    assert h.value == -7
    assert lib.rt_denoise_halo(3, 1, 1, None) == 1 and "NULL" in lib.rt_last_error().decode()
