"""CPU checks of the volume entry points: arguments are rejected before anything touches the device."""
import ctypes

import pytest


@pytest.fixture(scope="module")
def lib():
    from wavelets_b200.build import build_library
    build_library()
    from wavelets_b200 import _lib
    return _lib.load()


def test_volume_scratch_and_workspace_sizes(lib):
    assert lib.wb_volume_scratch_bytes(0, 4, 8, 8, 0) == 0
    assert lib.wb_volume_scratch_bytes(0, 4, 8, 8, 1) == 4 * 8 * 8 * 4            # the slice smooth only
    assert lib.wb_volume_scratch_bytes(1, 4, 8, 8, 3) == 3 * 4 * 8 * 8 * 8        # + two ping-pong smooth volumes
    # the whole volume is one frame of the MAD estimate and of the moments
    assert lib.wb_wow_cascade_volume_workspace_bytes(0, 4, 8, 8) == lib.wb_wow_cascade_workspace_bytes(0, 1, 256)


def test_scale_and_transform_volume_validation(lib):
    ok, other, tmp = ctypes.c_void_p(16), ctypes.c_void_p(32), ctypes.c_void_p(48)

    def scale(in_=ok, out_c=other, out_w=None, tmp_=tmp, D=4, scale_=0, taps=5, dtype=0):
        return lib.wb_atrous_scale_volume(in_, out_c, out_w, tmp_, D, 8, 8, scale_, taps, dtype, None)
    assert scale(dtype=3) == -1
    assert scale(taps=4) == -2
    assert scale(D=0) == -3
    assert scale(D=65536) == -3
    assert scale(scale_=31) == -4
    assert scale(in_=None) == -5
    assert scale(tmp_=None) == -5
    assert scale(out_c=None) == -5                             # nothing to write
    assert scale(out_c=ok) == -5                               # in place
    assert scale(tmp_=other) == -5                             # the slice smooth would overwrite c_{s+1}
    assert scale(out_c=other, out_w=other) == -5

    def transform(in_=ok, planes=other, scratch=tmp, levels=2, dtype=0):
        return lib.wb_atrous_transform_volume(in_, planes, scratch, 4, 8, 8, levels, 5, dtype, None)
    assert transform(dtype=2) == -1
    assert transform(levels=-1) == -4
    assert transform(levels=31) == -4
    assert transform(in_=None) == -5
    assert transform(planes=None) == -5
    assert transform(scratch=None) == -5


def test_wow_cascade_volume_validation(lib):
    ok = ctypes.c_void_p(16)
    arr = (ctypes.c_double * 3)(1.0, 1.0, 1.0)
    ws = lib.wb_wow_cascade_volume_workspace_bytes(0, 4, 8, 8)

    def call(n_scales=2, taps=5, dtype=0, planes=ok, scratch=ok, recon=ok, weights=arr, estimate=0, noise_dev=None,
             noise_map=None, zstride=0, workspace=ok, ws_bytes=ws, D=4):
        return lib.wb_wow_cascade_volume(ok, planes, scratch, recon, D, 8, 8, n_scales, taps, dtype, weights, arr, arr,
                                         1, 1, 0.0, noise_dev, estimate, noise_map, zstride, workspace, ws_bytes, None)
    assert call(dtype=5) == -1
    assert call(taps=7) == -2
    assert call(D=0) == -3
    assert call(n_scales=-1) == -4
    assert call(n_scales=31) == -4
    assert call(planes=None) == -5
    assert call(scratch=None) == -5                            # needed as soon as there is a scale
    assert call(recon=None) == -5
    assert call(weights=None) == -5
    assert call(workspace=None) == -5
    assert call(estimate=1) == -5                              # an estimate needs somewhere to go
    assert call(ws_bytes=ws - 1) == -6
    assert call(noise_map=ok, zstride=-1) == -6
    assert call(noise_map=ok, zstride=63) == -6                # slices of a full map are H * W apart at least
    assert call(noise_map=ok, estimate=1, noise_dev=ok) == -6  # a map and an estimate exclude each other


def test_wow_volume_route_selection():
    """The volume route covers plain volumes with h == 0 and no preserve_variance; the noise is classified as
    Coefficients._noise_arg classifies it (numbers and one-element tensors are scalars, everything else a map)."""
    import numpy as np
    import torch

    from wavelets_b200 import utils
    shape = (3, 4, 5)
    nz, zs, kept = utils._volume_noise(None, shape, torch.float32, "cpu", True)
    assert nz is None and kept is None
    nz, zs, kept = utils._volume_noise(2.5, shape, torch.float32, "cpu", True)
    assert nz.host == 2.5 and nz.map is None and kept == 2.5
    nz, zs, kept = utils._volume_noise(np.array(1.5), shape, torch.float32, "cpu", True)
    assert nz.host == 1.5
    nz, zs, kept = utils._volume_noise(torch.tensor([0.5]), shape, torch.float32, "cpu", True)
    assert nz.host == 0.5
    m = np.ones((4, 5))
    nz, zs, kept = utils._volume_noise(m, shape, torch.float32, "cpu", True)
    assert zs == 0 and tuple(nz.map.shape) == (4, 5) and tuple(kept.shape) == shape
    nz, zs, kept = utils._volume_noise(m, shape, torch.float32, "cpu", False)
    assert kept is m                                           # an unused map stays as given
    full = torch.ones(shape, dtype=torch.float64)
    nz, zs, kept = utils._volume_noise(full, shape, torch.float32, "cpu", True)
    assert zs == 20 and nz.map.dtype == torch.float32 and kept is full
    with pytest.raises(ValueError):
        utils._volume_noise(np.ones((2, 5)), shape, torch.float32, "cpu", True)
    with pytest.raises(TypeError):
        utils._volume_noise([1.0], shape, torch.float32, "cpu", True)
