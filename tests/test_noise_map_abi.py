"""CPU checks of the noise-map entry points: arguments are rejected before anything touches the device."""
import ctypes

import pytest


@pytest.fixture(scope="module")
def lib():
    from wavelets_b200.build import build_library
    build_library()
    from wavelets_b200 import _lib
    return _lib.load()


def test_whiten_scale_map_validation(lib):
    w, o, m = ctypes.c_void_p(16), ctypes.c_void_p(32), ctypes.c_void_p(48)

    def call(w=w, o=o, m=m, map_pitch=64, map_bstride=0, sigma=3.0, dtype=0, taps=5, scale=0):
        return lib.wb_wow_whiten_scale_map(w, o, m, 1, 16, 64, 64, 0, 64, 0, map_pitch, map_bstride, scale, taps, dtype,
                                           1, sigma, 1.0, 1.0, None)
    assert call(sigma=0.0) == -6  # unthresholded scales take wb_wow_whiten_scale with sig_mode 0
    assert call(map_pitch=63) == -6
    assert call(map_bstride=-1) == -6
    assert call(m=None) == -5
    assert call(m=o) == -5
    assert call(o=w) == -5
    assert call(dtype=7) == -1
    assert call(taps=4) == -2
    assert call(scale=31) == -4


def test_cascade_map_validation(lib):
    ok = ctypes.c_void_p(16)
    arr = (ctypes.c_double * 3)(1.0, 1.0, 1.0)
    ws = lib.wb_wow_cascade_workspace_bytes(0, 1, 64)

    def call(noise_map=ok, map_pitch=8, map_bstride=0, n_scales=2, ws_bytes=ws, planes=ok):
        return lib.wb_wow_cascade_map(ok, 8, 0, planes, ok, ok, 1, 8, 8, n_scales, 5, 0, arr, arr, arr, None, 1,
                                      noise_map, map_pitch, map_bstride, ok, ws_bytes, None)
    assert call(noise_map=None) == -5
    assert call(map_pitch=7) == -6
    assert call(map_bstride=-64) == -6
    assert call(n_scales=0) == -4
    assert call(planes=None) == -5
    assert call(ws_bytes=16) == -6
