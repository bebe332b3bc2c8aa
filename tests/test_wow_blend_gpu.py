"""wow() with the gamma blend (h > 0) and preserve_variance as one library call (wb_wow_cascade_blend), and the same
options in wow_batch and wow_stream.

The reference is the element-wise route that wow() took before: the transform, then _wow_general plane by plane (it
stays in the tree for Coefficients input).  Results must be bit-identical to it -- recon, every plane and the noise --
so the comparisons view the arrays as integers: NaN, inf and -0.0 count."""

import numpy as np
import pytest
import torch

from oracle import atrous_oracle as orc

pytestmark = pytest.mark.gpu


def _bits(t):
    return t.view(torch.int32 if t.dtype == torch.float32 else torch.int64)


def _assert_bitwise(a, b, msg=""):
    assert a.shape == b.shape and a.dtype == b.dtype, (msg, a.shape, b.shape, a.dtype, b.dtype)
    eq = _bits(a) == _bits(b)
    assert bool(eq.all()), (msg, int((~eq).sum()), a[~eq][:4].tolist(), b[~eq][:4].tolist())


def _assert_same_noise(a, b, msg=""):
    if isinstance(a, torch.Tensor) or isinstance(b, torch.Tensor):
        assert isinstance(a, torch.Tensor) and isinstance(b, torch.Tensor), (msg, type(a), type(b))
        _assert_bitwise(a, b, msg)
    elif isinstance(a, np.ndarray) or isinstance(b, np.ndarray):
        assert np.array_equal(np.asarray(a), np.asarray(b)), msg
    else:
        assert (a is None and b is None) or a == b, (msg, a, b)


def _parent_route(img, kw):
    """wow(img, **kw) the way the parent commit computed it (utils.py: the `general` branch of wow())."""
    import wavelets_b200 as wb
    from wavelets_b200 import utils
    kw = dict(kw)
    sf = kw.pop("scaling_function", wb.B3spline)
    h = kw.get("h", 0)
    n_scales, sigma_bilateral, wts, dns = utils._wow_plan(img.shape, sf, kw.get("n_scales"), kw.get("weights", []),
                                                          kw.get("denoise_coefficients", []), kw.get("bilateral"), h=h)
    co = wb.AtrousTransform(sf, bilateral=sigma_bilateral, bilateral_scaling=kw.get("bilateral_scaling", False))(
        img, n_scales)
    co.noise = kw.get("noise")
    recon, co = utils._wow_general(co, kw.get("weights", []), kw.get("whitening", True),
                                   kw.get("denoise_coefficients", []), kw.get("bilateral"),
                                   kw.get("soft_threshold", True), kw.get("preserve_variance", False),
                                   kw.get("gamma", 3.2), kw.get("gamma_min"), kw.get("gamma_max"), h,
                                   plan=(n_scales, wts, dns))
    return recon, co


def _frame(shape, dt, seed=3, flux=0.05):
    return orc.solar_like(max(shape), seed=seed, flux=flux, dtype=dt)[:shape[0], :shape[1]].copy()


def _photon_map(frame, gain=1.5, read=3.0):
    return np.sqrt(gain * np.maximum(frame, 0) + read ** 2).astype(frame.dtype)


def _quantiles(shape, dt):
    f = _frame(shape, dt)
    return float(np.quantile(f, 0.2)), float(np.quantile(f, 0.8))


LO, HI = _quantiles((256, 256), np.float32)
DEN = {"denoise_coefficients": [4, 2]}

# (shape, dtype, kwargs); "noise" values that are strings are built per case (see _noise)
WOW_CASES = [
    ((256, 256), np.float32, dict(h=0.4, denoise_coefficients=[5, 2])),                  # MAD estimate at scale 0
    ((256, 256), np.float32, dict(h=1, denoise_coefficients=[3, 2, 1])),                 # no whitening (h >= 1)
    ((256, 256), np.float32, dict(h=1)),                                                  # L = 0
    ((256, 256), np.float32, dict(h=1.5, n_scales=3)),
    ((256, 256), np.float32, dict(preserve_variance=True)),
    ((256, 256), np.float32, dict(preserve_variance=True, h=0.25, denoise_coefficients=[4, 2], weights=[1.5, 0.5])),
    ((256, 256), np.float32, dict(preserve_variance=True, h=-0.5, weights=[1.5, 0.5, 2])),  # h < 0: no blend
    ((256, 256), np.float32, dict(whitening=False, h=0.5, denoise_coefficients=[4, 2], weights=[0.5, 2])),
    ((256, 256), np.float32, dict(whitening=False, preserve_variance=True, h=0.5, weights=[0.5, 1, 2])),
    ((256, 256), np.float32, dict(whitening=False, preserve_variance=True, denoise_coefficients=[3])),
    ((256, 256), np.float32, dict(h=0.3, gamma_min=LO)),
    ((256, 256), np.float32, dict(h=0.3, gamma_max=HI)),
    ((256, 256), np.float32, dict(h=0.3, gamma_min=LO, gamma_max=HI)),
    ((256, 256), np.float32, dict(h=0.3, gamma_min=LO, gamma_max=HI, gamma=2.5, preserve_variance=True)),
    ((256, 256), np.float32, dict(h=0.5, gamma=2.5, **DEN)),
    ((256, 256), np.float32, dict(h=0.5, gamma=2, **DEN)),
    ((256, 256), np.float32, dict(h=0.5, gamma=1, **DEN)),
    ((256, 256), np.float32, dict(h=0.5, gamma=2, gamma_min=LO, gamma_max=HI)),
    ((256, 256), np.float32, dict(h=0.5, denoise_coefficients=[0, 3])),                  # MAD at a first threshold on 1
    ((256, 256), np.float32, dict(h=0.5, preserve_variance=True, denoise_coefficients=[0, 3, 1])),
    ((256, 256), np.float32, dict(h=0.5, noise="host", **DEN)),
    ((256, 256), np.float32, dict(h=0.5, noise="host", soft_threshold=False, **DEN)),
    ((256, 256), np.float32, dict(h=0.5, noise="host_zero", **DEN)),
    ((256, 256), np.float32, dict(h=0.5, noise="device", preserve_variance=True, **DEN)),
    ((256, 256), np.float32, dict(h=0.5, noise="device_zero", **DEN)),
    ((256, 256), np.float32, dict(h=0.5, noise="map", **DEN)),
    ((256, 256), np.float32, dict(h=0.5, noise="map", soft_threshold=False, preserve_variance=True, **DEN)),
    ((256, 256), np.float32, dict(h=0.5, noise="map_tensor", whitening=False, **DEN)),
    ((256, 256), np.float32, dict(h=0.5, noise="map", whitening=False, soft_threshold=False, **DEN)),
    ((256, 256), np.float32, dict(h=0.5, bilateral=1, **DEN)),
    ((192, 320), np.float32, dict(h=0.3, bilateral=[1, 2], bilateral_scaling=True, preserve_variance=True,
                                  denoise_coefficients=[0, 3], soft_threshold=False)),
    ((160, 160), np.float64, dict(h=0.5, preserve_variance=True, scaling_function="triangle", **DEN)),
    ((128, 128), np.float64, dict(h=0.4, bilateral=1, noise="map", **DEN)),
    ((96, 201), np.float32, dict(h=0.5, preserve_variance=True, denoise_coefficients=[3, 1])),   # generic kernels
    ((64, 2560), np.float64, dict(h=0.5, denoise_coefficients=[2], soft_threshold=False)),        # fp64 wide rows
    ((64, 2560), np.float64, dict(h=0.5, preserve_variance=True, gamma=2.5, gamma_min=LO)),
]


def _noise(kind, frame, device="cuda"):
    if kind == "host":
        return 1.25
    if kind == "host_zero":
        return 0.0
    if kind == "device":
        return torch.tensor([1.25], dtype=torch.float64, device=device)
    if kind == "device_zero":
        return torch.zeros(1, dtype=torch.float64, device=device)
    if kind == "map":
        return _photon_map(frame)
    if kind == "map_tensor":
        return torch.from_numpy(_photon_map(frame)).to(device)
    return kind


def _check_against_parent(img, kw, msg):
    import wavelets_b200 as wb
    ref_kw, new_kw = dict(kw), dict(kw)
    sf = {"triangle": wb.Triangle, "b3spline": wb.B3spline}[kw.get("scaling_function", "b3spline")]
    ref_kw["scaling_function"] = new_kw["scaling_function"] = sf
    frame = img.cpu().numpy()
    if isinstance(kw.get("noise"), str):
        ref_kw["noise"] = _noise(kw["noise"], frame)
        new_kw["noise"] = _noise(kw["noise"], frame)
    r_ref, co_ref = _parent_route(img, ref_kw)
    r, co = wb.wow(img, **new_kw)
    _assert_bitwise(r, r_ref, (msg, "recon"))
    _assert_bitwise(co.data, co_ref.data, (msg, "planes"))
    _assert_same_noise(co._noise, co_ref._noise, (msg, "noise"))
    return r, co


@pytest.mark.parametrize("case", range(len(WOW_CASES)))
def test_wow_blend_equals_parent_route(case):
    shape, dt, kw = WOW_CASES[case]
    img = torch.from_numpy(_frame(shape, dt)).cuda()
    _check_against_parent(img, kw, case)


def test_wow_blend_full_size():
    img = torch.from_numpy(orc.solar_like(4096, seed=7, flux=1, dtype=np.float32)).cuda()
    _check_against_parent(img, dict(h=0.9, denoise_coefficients=[5, 2]), "4096")


@pytest.mark.parametrize("kw", [dict(h=0.5, preserve_variance=True), dict(h=0.5, denoise_coefficients=[3]),
                                dict(h=0.5, gamma_min=2.0, gamma_max=2.0), dict(h=0.5, gamma=1, whitening=False),
                                dict(h=1), dict(preserve_variance=True, whitening=False)])
@pytest.mark.parametrize("dt", [np.float32, np.float64])
def test_wow_blend_constant_frame(kw, dt):
    """Zero std and a zero gamma range: 1e-15 divisors, 0 / 0 and inf * 0 must give the same NaN / inf bits."""
    img = torch.full((128, 192), 2.0, dtype=torch.float32 if dt == np.float32 else torch.float64, device="cuda")
    r, _ = _check_against_parent(img, kw, "constant")
    if kw.get("h", 0) > 0 and kw.get("gamma_min") is None:
        assert bool(torch.isnan(r).all())


def test_wow_blend_returns_array_and_gamma_zero_raises():
    import wavelets_b200 as wb
    frame = _frame((128, 128), np.float32)
    r, co = wb.wow(frame, h=0.5, preserve_variance=True)
    assert isinstance(r, np.ndarray) and r.dtype == np.float32 and len(co) == len(co.data)
    with pytest.raises(ZeroDivisionError):
        wb.wow(frame, h=0.5, gamma=0)


# ------------------------------------------------------------------------------------------------------------------
# wow_batch / wow_stream against single wow() calls
# ------------------------------------------------------------------------------------------------------------------
BATCH_KW = [dict(h=0.5, preserve_variance=True, denoise_coefficients=[4, 2]),
            dict(h=0.4, gamma=2.5, bilateral=1, denoise_coefficients=[3, 1]),
            dict(h=1, denoise_coefficients=[3, 2], soft_threshold=False, weights=[0.5, 2]),
            dict(h=0.3, gamma_min=LO, whitening=False, denoise_coefficients=[0, 2])]


def _stack(n, shape=(192, 256), dt=np.float32):
    return np.stack([_frame(shape, dt, seed=s) for s in range(n)])


@pytest.mark.parametrize("kw", range(len(BATCH_KW)))
def test_wow_batch_blend_equals_single_calls(kw):
    import wavelets_b200 as wb
    kw = BATCH_KW[kw]
    frames = _stack(3)
    maps = np.stack([_photon_map(f) for f in frames])
    vec = np.array([0.5, 1.0, 2.0])
    forms = [("none", None, lambda i: None), ("scalar", 1.5, lambda i: 1.5), ("vec", vec, lambda i: float(vec[i])),
             ("shared", maps[0], lambda i: maps[0]), ("per_frame", torch.from_numpy(maps).cuda(), lambda i: maps[i])]
    for name, noise, single in forms:
        recon, planes, _ = wb.wow_batch(frames, noise=noise, **kw)
        for i in range(len(frames)):
            r, co = wb.wow(frames[i], noise=single(i), **kw)
            _assert_bitwise(recon[i], torch.from_numpy(r).cuda(), (name, i, "recon"))
            _assert_bitwise(planes[i], co.data, (name, i, "planes"))


STREAM_KW = BATCH_KW + [dict(h=1), dict(preserve_variance=True, noise=0.8)]


@pytest.mark.parametrize("depth", [1, 2, 3])
def test_wow_stream_blend_equals_single_calls(depth, monkeypatch):
    import wavelets_b200 as wb
    from wavelets_b200 import utils
    frames = _stack(4)
    maps = np.stack([_photon_map(f) for f in frames])
    singles = []
    cases = [(kw, kw.get("noise"), lambda i, kw=kw: kw.get("noise")) for kw in STREAM_KW]
    cases.append((dict(BATCH_KW[0], noise=maps), maps, lambda i: maps[i]))
    for kw, _, single in cases:
        kw_single = {k: v for k, v in kw.items() if k != "noise"}
        singles.append([wb.wow(frames[i], noise=single(i), **kw_single)[0] for i in range(len(frames))])

    def no_per_frame_fallback(*args, **kwargs):
        raise AssertionError("wow_stream() must not call wow() per frame")
    monkeypatch.setattr(utils, "wow", no_per_frame_fallback)
    for (kw, _, _), ref in zip(cases, singles):
        for inp in (frames, torch.from_numpy(frames).pin_memory()):
            out = utils.wow_stream(inp, depth=depth, **kw)
            out = out if isinstance(out, np.ndarray) else out.numpy()
            for i in range(len(frames)):
                assert np.array_equal(out[i].view(np.int32), ref[i].view(np.int32)), (kw, depth, i)


# ------------------------------------------------------------------------------------------------------------------
# Only the library's kernels run
# ------------------------------------------------------------------------------------------------------------------
def test_wow_blend_launches_only_library_kernels():
    import wavelets_b200 as wb
    from torch.profiler import ProfilerActivity, profile
    img = torch.from_numpy(_frame((512, 512), np.float32)).cuda()
    wb.wow(img, h=0.5, preserve_variance=True)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        wb.wow(img, h=0.5, preserve_variance=True)
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type.name == "CUDA"]
    kernels = [k for k in names if not k.startswith(("Memcpy", "Memset"))]
    assert kernels, names
    foreign = sorted({k for k in kernels if "wb::" not in k and "_ZN2wb" not in k})
    assert not foreign, foreign
