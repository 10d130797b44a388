"""CPU-side checks of the moments sink ABI (include/rt_b200.h): the ctypes mirror of rt_path_moments_sink has the C
layout, and the library that exports the new entries reports the version that introduced them."""
import ctypes as C
import os

import pytest


@pytest.fixture(scope="module")
def native():
    from ray_tracer_v1_b200 import _native
    if not os.path.exists(_native.LIB_PATH):
        _native.build()
    return _native


def test_moments_sink_layout_and_version(native):
    assert C.sizeof(native.PathMomentsSink) == native.RT_MAX_PEERS * 8 + 8
    assert native.PathMomentsSink.var.offset == native.RT_MAX_PEERS * 8
    lib = native.load_symbols()
    assert lib.rt_version() >= 102
    for name in ("rt_render_path_sink_moments", "rt_resolve_clear_moments"):
        assert name in native.SIGNATURES and hasattr(lib, name)
