"""CPU checks of wb_wow_cascade_blend: arguments are rejected before anything touches the device."""
import ctypes

import pytest


@pytest.fixture(scope="module")
def lib():
    from wavelets_b200.build import build_library
    build_library()
    from wavelets_b200 import _lib
    return _lib.load()


def test_cascade_blend_validation(lib):
    ok = ctypes.c_void_p(16)
    arr = (ctypes.c_double * 3)(1.0, 1.0, 1.0)
    ws = lib.wb_wow_cascade_blend_workspace_bytes(0, 1, 64)
    assert ws > lib.wb_wow_cascade_workspace_bytes(0, 1, 64)

    def call(gamma_plane=ok, n_scales=2, dtype=0, taps=5, planes=ok, scratch=ok, estimate=0, noise_dev=None, use_map=0,
             noise_map=None, map_pitch=8, map_bstride=0, h=0.5, gamma=3.2, ws_bytes=ws, workspace=ok):
        return lib.wb_wow_cascade_blend(ok, 8, 0, planes, scratch, ok, gamma_plane, 1, 8, 8, n_scales, taps, dtype, arr,
                                        arr, arr, None, 1, 0.0, noise_dev, estimate, use_map, noise_map, map_pitch,
                                        map_bstride, 1, 1, h, gamma, 0.0, 0, 0.0, 0, workspace, ws_bytes, None)
    assert call(gamma_plane=None) == -5                       # the blend needs the gamma plane
    assert call(gamma=0.0) == -6                              # 1 / gamma
    assert call(use_map=1) == -5                              # map flag set, no map
    assert call(use_map=1, noise_map=ok, map_pitch=7) == -6
    assert call(use_map=1, noise_map=ok, map_bstride=-1) == -6
    assert call(use_map=1, noise_map=ok, estimate=1, noise_dev=ok) == -6
    assert call(estimate=1) == -5                             # an estimate needs somewhere to go
    assert call(ws_bytes=lib.wb_wow_cascade_workspace_bytes(0, 1, 64)) == -6  # the plain cascade's is too short
    assert call(workspace=None) == -5
    assert call(dtype=7) == -1
    assert call(taps=4) == -2
    assert call(n_scales=-1) == -4
    assert call(n_scales=31) == -4
    assert call(planes=None) == -5
    assert call(scratch=None) == -5                           # scratch is needed as soon as there is a scale


def test_cascade_keeps_rejecting_zero_scales(lib):
    """n_scales == 0 is accepted by the blend route only; the whitening cascade still rejects it."""
    ok = ctypes.c_void_p(16)
    arr = (ctypes.c_double * 1)(1.0)
    ws = lib.wb_wow_cascade_workspace_bytes(0, 1, 64)
    assert lib.wb_wow_cascade(ok, 8, 0, ok, ok, ok, 1, 8, 8, 0, 5, 0, arr, arr, arr, None, 1, 0.0, None, 0, ok, ws,
                              None) == -4


def test_wow_batch_and_stream_take_the_blend_options():
    import inspect

    from wavelets_b200 import utils
    params = inspect.signature(utils.wow_batch).parameters
    for name, default in (("preserve_variance", False), ("gamma", 3.2), ("gamma_min", None), ("gamma_max", None),
                          ("h", 0)):
        assert params[name].default == default, name
    assert utils._blend_options(False, 3.2, None, None, 0) is None
    assert utils._blend_options(True, 0, None, None, 0) == (True, 0.0, None, None, 0.0)  # gamma unused without blend
    with pytest.raises(ZeroDivisionError):
        utils._blend_options(False, 0, None, None, 0.5)
