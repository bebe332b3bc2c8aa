"""Volumes (D, H, W) on wb_atrous_transform_volume / wb_wow_cascade_volume: bit-identical to the per-scale route they
replace (wb_atrous_scale + wb_atrous_axis for the transform, the element-wise loop _wow_nd for wow())."""
import numpy as np
import pytest
import torch

import wavelets_b200 as wb
from wavelets_b200 import utils, wavelets

pytestmark = pytest.mark.gpu

SF = {"triangle": wb.Triangle, "b3spline": wb.B3spline}
DT = {"f32": torch.float32, "f64": torch.float64}


def cube(shape, dtype, seed=0):
    g = torch.Generator().manual_seed(seed)
    base = torch.rand(shape, generator=g, dtype=torch.float64) * 4 + 1
    return (base + torch.randn(shape, generator=g, dtype=torch.float64) * 0.3).to(dtype).cuda()


def ref_transform(vol, sf, level):
    return wb.AtrousTransform(sf)._run_nd_reference(vol, level, sf(3))


# D in {1, 2, 3} puts every dilation at or beyond the depth (several reflections); W = 37 / 1025 break the 16-byte
# vectors of the slice and depth passes
TRANSFORM_SHAPES = [((1, 12, 16), 4), ((2, 9, 20), 4), ((3, 16, 12), 5), ((17, 15, 37), 5), ((64, 24, 32), 7),
                    ((5, 8, 1025), 3)]


@pytest.mark.parametrize("dt", DT)
@pytest.mark.parametrize("name", SF)
@pytest.mark.parametrize("shape,level", TRANSFORM_SHAPES)
def test_transform_volume_matches_reference(shape, level, name, dt):
    vol = cube(shape, DT[dt])
    sf = SF[name]
    got = wb.AtrousTransform(sf)(vol, level).data
    assert torch.equal(got, ref_transform(vol, sf, level))
    for s in range(level):
        assert torch.equal(wavelets._smooth_nd(vol, s, sf(3)), wavelets._smooth_nd_reference(vol, s, sf(3)))


def test_volume_callers_take_the_new_route():
    vol = cube((9, 16, 20), torch.float32)
    out = wb.convolution(vol, wb.B3spline(3), 2)
    assert torch.equal(out, wavelets._smooth_nd_reference(vol, 2, wb.B3spline(3)))
    got = utils.denoise(vol, [3, 1], noise=0.2)
    co = ref_transform(vol, wb.B3spline, 2)
    ref = wavelets.Coefficients(co, wb.B3spline(3))
    ref.noise = 0.2
    ref.denoise([3, 1])
    assert torch.equal(got, wavelets.synthesis(co.reshape(3, 1, -1)).reshape(vol.shape))


def ref_wow(vol, sf, noise, n_scales=None, weights=(), whitening=True, denoise_coefficients=(), soft_threshold=True):
    L, _, wts, dns = utils._wow_plan(vol.shape, sf, n_scales, list(weights), list(denoise_coefficients), None,
                                     n_dims=3)
    co = wavelets.Coefficients(ref_transform(vol, sf, L), sf(3), None)
    co.noise = noise
    recon = utils._wow_nd(co, wts, dns, whitening, soft_threshold, False, 3.2, None, None, 0,
                          smooth=wavelets._smooth_nd_reference)
    return recon, co


def same_noise(a, b):
    if isinstance(a, torch.Tensor) or isinstance(b, torch.Tensor):
        return torch.equal(torch.as_tensor(a).cuda(), torch.as_tensor(b).cuda())
    if isinstance(a, np.ndarray):
        return a is b or np.array_equal(a, b)
    return a == b


OPTIONS = {
    "default": {},
    "weights": dict(weights=[1.5, 0.7, 2.0, 0.3]),
    "no_whitening": dict(whitening=False, weights=[0.1, 3.0], denoise_coefficients=[2, 1]),
    "soft": dict(denoise_coefficients=[3, 2, 1]),
    "hard": dict(denoise_coefficients=[3, 2, 1], soft_threshold=False),
    "first_and_fourth": dict(denoise_coefficients=[0, 3]),
    "hard_no_whitening": dict(whitening=False, denoise_coefficients=[0, 3], soft_threshold=False),
}
NOISES = ["none", "scalar", "device", "map_hw", "map_full"]


def make_noise(kind, shape, dtype):
    d, h, w = shape
    g = np.random.default_rng(1)
    if kind == "none":
        return None
    if kind == "scalar":
        return 0.05
    if kind == "device":
        return torch.tensor([0.04], dtype=torch.float64, device="cuda")
    if kind == "map_hw":
        return (g.random((h, w)) * 0.05 + 0.01).astype(np.float64)
    return torch.as_tensor(g.random(shape) * 0.05 + 0.01).to(dtype).cuda()


def check_wow(vol, sf, noise, **opts):
    recon, co = wb.wow(vol, scaling_function=sf, noise=noise, **opts)
    ref_recon, ref_co = ref_wow(vol, sf, noise, **opts)
    assert torch.equal(co.data, ref_co.data)
    assert torch.equal(recon, ref_recon)
    assert same_noise(co._noise, ref_co._noise)


@pytest.mark.parametrize("dt", DT)
@pytest.mark.parametrize("name", SF)
@pytest.mark.parametrize("opt", OPTIONS)
@pytest.mark.parametrize("noise", NOISES)
def test_wow_volume_matches_reference(noise, opt, name, dt):
    shape = (17, 40, 48)
    vol = cube(shape, DT[dt], seed=3)
    check_wow(vol, SF[name], make_noise(noise, shape, DT[dt]), **OPTIONS[opt])


# odd H / W, a width outside the 16-byte vectors, 64 slices, and D = 3 where a Triangle plans no scale at all
@pytest.mark.parametrize("dt", DT)
@pytest.mark.parametrize("shape,name", [((64, 33, 35), "b3spline"), ((20, 31, 1025), "triangle"),
                                        ((3, 16, 16), "triangle"), ((40, 64, 64), "triangle")])
def test_wow_volume_shapes(shape, name, dt):
    vol = cube(shape, DT[dt], seed=5)
    check_wow(vol, SF[name], None, denoise_coefficients=[2, 1])
    check_wow(vol, SF[name], make_noise("map_hw", shape, DT[dt]), denoise_coefficients=[0, 3], soft_threshold=False)


def test_wow_volume_numpy_in_numpy_out():
    vol = cube((12, 20, 24), torch.float64, seed=7)
    recon, co = wb.wow(vol.cpu().numpy(), denoise_coefficients=[1])
    ref_recon, ref_co = ref_wow(vol, wb.B3spline, None, denoise_coefficients=[1])
    assert isinstance(recon, np.ndarray) and np.array_equal(recon, ref_recon.cpu().numpy())
    assert co.noise == ref_co.noise


def test_wow_volume_launches_library_kernels_only():
    vol = cube((32, 64, 64), torch.float32, seed=9)
    wb.wow(vol, denoise_coefficients=[3, 1])
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        wb.wow(vol, denoise_coefficients=[3, 1], weights=[1, 2])
        torch.cuda.synchronize()
    kernels = {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA
               and not e.name.startswith(("Memcpy", "Memset", "cudaMemcpy", "cudaMemset"))}
    assert kernels
    assert all("wb::" in k for k in kernels), sorted(kernels)


def test_wow_volume_peak_memory():
    import wavelets_b200._lib as L
    shape = (32, 256, 256)
    vol = cube(shape, torch.float32, seed=11)
    lib = L.load()
    n_scales = 4
    vol_bytes = vol.numel() * 4
    declared = (lib.wb_volume_scratch_bytes(0, *shape, n_scales) + lib.wb_wow_cascade_volume_workspace_bytes(0, *shape)
                + (n_scales + 1) * vol_bytes + vol_bytes)  # scratch, workspace, planes, reconstruction
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    out = wb.wow(vol, n_scales=n_scales, denoise_coefficients=[3, 1])
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    del out
    assert peak <= declared + (4 << 20), (peak, declared)
