"""Per-pixel noise maps on the device: the map mode of the whitening kernel (wb_wow_whiten_scale_map), the map cascade
(wb_wow_cascade_map) behind wow(img, noise=map), and the (B,) / (H, W) / (B, H, W) noise of wow_batch and wow_stream.

The map mode must equal, bit for bit, the composition it replaces: the mode-0 whitening, wb_significance with the map
and the float64 product of the two.  Bitwise comparisons view the planes as integers, so NaN payloads and -0.0 count."""

import numpy as np
import pytest
import torch

from oracle import atrous_oracle as orc

pytestmark = pytest.mark.gpu


def _lib():
    from wavelets_b200 import _lib as L
    return L, L.load(require_cuda=True)


def _bits(t):
    return t.view(torch.int32 if t.dtype == torch.float32 else torch.int64)


def _assert_bitwise(a, b, msg=""):
    assert a.shape == b.shape and a.dtype == b.dtype, msg
    eq = _bits(a) == _bits(b)
    assert bool(eq.all()), (msg, int((~eq).sum()), a[~eq][:4].tolist(), b[~eq][:4].tolist())


def _sf(name):
    import wavelets_b200 as wb
    return {"b3spline": wb.B3spline, "triangle": wb.Triangle}[name]


@pytest.fixture(scope="module")
def maps_and_planes():
    """Raw detail planes and noise maps with zeros, negative entries and zero coefficients (0 / 0 thresholds)."""
    def make(b, h, w, dt, seed):
        g = torch.Generator(device="cpu").manual_seed(seed)
        raw = torch.randn((b, h, w), generator=g, dtype=torch.float64) * 3
        raw[:, ::7, ::5] = 0.0
        nmap = torch.rand((b, h, w), generator=g, dtype=torch.float64) * 2 + 0.05
        nmap[:, ::11, ::3] = 0.0
        nmap[:, 5::13, 1::4] *= -1
        return raw.to(dt).cuda(), nmap.to(dt).cuda()
    return make


def _composition(raw, nmap_frames, s, taps, soft, sigma, sigma_e, weight):
    """The unfused route: K3 with sig_mode 0, wb_significance with the map, the float64 product rounded once."""
    L, lib = _lib()
    b, h, w = raw.shape
    tmp = torch.empty_like(raw)
    code = L.dtype_code(raw.dtype)
    st = L.stream_ptr(raw.device)
    L.check(lib.wb_wow_whiten_scale(raw.data_ptr(), tmp.data_ptr(), b, h, w, w, h * w, w, h * w, s, taps, code, 0, 0.0,
                                    1.0, 0.0, None, float(weight), st))
    out = torch.empty_like(raw)
    for f in range(b):
        sig = torch.empty((h, w), dtype=torch.float64 if soft else torch.uint8, device=raw.device)
        L.check(lib.wb_significance(raw[f].data_ptr(), h * w, code, float(sigma), float(sigma_e), 0.0, None,
                                    nmap_frames[f].data_ptr(), 1 if soft else 0, sig.data_ptr(), st))
        out[f] = (tmp[f].to(torch.float64) * sig.to(torch.float64)).to(raw.dtype)
    return out


def _map_kernel(raw, nmap, map_pitch, map_bstride, s, taps, soft, sigma, sigma_e, weight, out=None):
    L, lib = _lib()
    b, h, w = raw.shape
    out = torch.empty_like(raw) if out is None else out
    L.check(lib.wb_wow_whiten_scale_map(raw.data_ptr(), out.data_ptr(), nmap.data_ptr(), b, h, w, w, h * w, w, h * w,
                                        map_pitch, map_bstride, s, taps, L.dtype_code(raw.dtype), 1 if soft else 0,
                                        float(sigma), float(sigma_e), float(weight), L.stream_ptr(raw.device)))
    return out


KERNEL_CASES = [(torch.float32, 128, 96), (torch.float32, 201, 48), (torch.float32, 1024, 40),
                (torch.float32, 2304, 24), (torch.float32, 4096, 20), (torch.float32, 6000, 12),
                (torch.float64, 128, 64), (torch.float64, 1024, 24), (torch.float64, 3000, 12)]


@pytest.mark.parametrize("dt,w,h", KERNEL_CASES)
@pytest.mark.parametrize("sf", ["b3spline", "triangle"])
def test_map_kernel_equals_composition(maps_and_planes, dt, w, h, sf):
    """Every dilation up to c * d > W, soft and hard, batch 1 and 3, shared and per-frame maps, maps with zero and
    negative entries; W = 201 also reads its map through an odd pitch (generic kernels)."""
    taps = _sf(sf)(2).taps_code
    c = taps // 2
    raw, nmap = maps_and_planes(3, h, w, dt, seed=w + taps)
    odd = None
    if w == 201:
        odd = torch.zeros((3, h, w + 1), dtype=dt, device="cuda")
        odd[:, :, :w] = nmap
    s_max = 0
    while c * (1 << s_max) <= w:
        s_max += 1
    for s in range(s_max + 1):
        for soft in (True, False):
            sigma, sigma_e, weight = 3.0, 0.7 + 0.01 * s, 1.25
            for batch in (1, 3):
                r = raw[:batch].contiguous()
                # one map per frame
                ref = _composition(r, [nmap[f] for f in range(batch)], s, taps, soft, sigma, sigma_e, weight)
                if odd is None:
                    got = _map_kernel(r, nmap, w, h * w, s, taps, soft, sigma, sigma_e, weight)
                else:
                    got = _map_kernel(r, odd, w + 1, h * (w + 1), s, taps, soft, sigma, sigma_e, weight)
                _assert_bitwise(got, ref, (dt, w, sf, s, soft, batch, "per-frame"))
                # one map for every frame
                ref = _composition(r, [nmap[0]] * batch, s, taps, soft, sigma, sigma_e, weight)
                got = _map_kernel(r, nmap[0], w, 0, s, taps, soft, sigma, sigma_e, weight)
                _assert_bitwise(got, ref, (dt, w, sf, s, soft, batch, "shared"))


# ------------------------------------------------------------------------------------------------------------------
# wow(img, noise=map) against the route of the parent: transform, then per thresholded scale K3 mode 0, the
# significance map and the float64 product; per unthresholded scale K3; the residual rescale and the synthesis
# ------------------------------------------------------------------------------------------------------------------
def _parent_map_route(img, noise, scaling_function, n_scales=None, weights=(), denoise_coefficients=(), bilateral=None,
                      bilateral_scaling=False, soft_threshold=True, whitening=True):
    import wavelets_b200 as wb
    from wavelets_b200 import utils
    from wavelets_b200.wavelets import _Noise, plane_moments, synthesis
    L_, lib = _lib()
    n_scales, sigma_bilateral, wts, dns = utils._wow_plan(img.shape, scaling_function, n_scales, list(weights),
                                                          list(denoise_coefficients), bilateral)
    co = wb.AtrousTransform(scaling_function, bilateral=sigma_bilateral, bilateral_scaling=bilateral_scaling)(img,
                                                                                                            n_scales)
    co.noise = noise
    data = co.data
    sf = co.scaling_function
    tmp = torch.empty_like(data[0])
    for s in range(n_scales):
        d, wt = dns[s], wts[s]
        plane = data[s]
        if not whitening:
            co._denoise_plane(lib, s, d, wt, soft_threshold)
            continue
        if d != 0:
            sig = co.significance(d, s, soft_threshold=soft_threshold)
            utils._whiten_scale(lib, plane, tmp, s, sf, 0, 0.0, 1.0, _Noise(), wt)
            plane.copy_((tmp.to(torch.float64) * sig.to(torch.float64)).to(plane.dtype))
        else:
            utils._whiten_scale(lib, plane, tmp, s, sf, 0, 0.0, 1.0, _Noise(), wt)
            plane.copy_(tmp)
    last = data[n_scales]
    if whitening:
        mom = plane_moments(last)
        L_.check(lib.wb_residual_rescale(last.data_ptr(), last.numel(), 1, 0, L_.dtype_code(last.dtype), mom.data_ptr(),
                                         float(wts[n_scales]), L_.stream_ptr(last.device)))
    elif wts[n_scales] != 1:
        last.mul_(wts[n_scales])
    return synthesis(data), data


def _photon_map(frame, gain=1.5, read=3.0):
    return np.sqrt(gain * np.maximum(frame, 0) + read ** 2).astype(frame.dtype)


WOW_MAP_CASES = [((256, 256), np.float32, {"denoise_coefficients": [5, 2]}),
                 ((256, 256), np.float32, {"denoise_coefficients": [5, 2], "soft_threshold": False}),
                 ((256, 256), np.float32, {"bilateral": 1, "denoise_coefficients": [5, 2]}),
                 ((192, 320), np.float32, {"bilateral": [1, 2], "denoise_coefficients": [0, 3], "bilateral_scaling": True,
                                           "soft_threshold": False}),
                 ((130, 1024), np.float32, {"denoise_coefficients": [4, 0, 2], "weights": [0.5, 2, 1.5]}),
                 ((128, 2304), np.float32, {"denoise_coefficients": [4]}),
                 ((64, 6000), np.float32, {"denoise_coefficients": [3, 1]}),                       # beyond the fused kernel
                 ((96, 201), np.float32, {"denoise_coefficients": [3, 1]}),                        # W % 4 != 0
                 ((160, 160), np.float64, {"denoise_coefficients": [5, 2], "scaling_function": "triangle"}),
                 ((64, 2560), np.float64, {"denoise_coefficients": [2], "soft_threshold": False}),
                 ((128, 128), np.float64, {"bilateral": 1, "denoise_coefficients": [4, 1]}),
                 ((160, 256), np.float32, {"denoise_coefficients": [4, 2], "whitening": False, "weights": [0.5, 2]})]


def _frame(shape, dt, seed=3, flux=0.05):
    return orc.solar_like(max(shape), seed=seed, flux=flux, dtype=dt)[:shape[0], :shape[1]].copy()


@pytest.mark.parametrize("case", range(len(WOW_MAP_CASES)))
def test_wow_map_equals_parent_route(case):
    import wavelets_b200 as wb
    shape, dt, kw = WOW_MAP_CASES[case]
    kw = dict(kw)
    sf = _sf(kw.pop("scaling_function", "b3spline"))
    img = torch.from_numpy(_frame(shape, dt)).cuda()
    nmap = torch.from_numpy(_photon_map(_frame(shape, dt))).cuda()
    r_ref, p_ref = _parent_map_route(img, nmap, sf, **kw)
    r, co = wb.wow(img, scaling_function=sf, noise=nmap, **kw)
    _assert_bitwise(r, r_ref, (case, "recon"))
    _assert_bitwise(co.data, p_ref, (case, "planes"))
    assert co.noise is nmap
    # wow() on existing coefficients with a map (the per-scale entry point)
    n_scales = len(p_ref) - 1
    co = wb.AtrousTransform(sf, bilateral=kw.get("bilateral"), bilateral_scaling=kw.get("bilateral_scaling", False))(
        img, n_scales)
    co.noise = nmap.cpu().numpy()
    okw = {k: v for k, v in kw.items() if k not in ("bilateral_scaling",)}
    r_co, co2 = wb.wow(co, **okw)
    assert co2 is co
    _assert_bitwise(r_co, r_ref, (case, "coefficients"))


def test_wow_map_full_size_bilateral():
    import wavelets_b200 as wb
    frame = orc.solar_like(4096, seed=7, flux=1, dtype=np.float32)
    img = torch.from_numpy(frame).cuda()
    nmap = torch.from_numpy(np.sqrt(frame) + 1).cuda()
    r_ref, p_ref = _parent_map_route(img, nmap, wb.B3spline, denoise_coefficients=[5, 2], bilateral=1)
    r, co = wb.wow(img, noise=nmap, denoise_coefficients=[5, 2], bilateral=1)
    _assert_bitwise(r, r_ref, "recon")
    _assert_bitwise(co.data, p_ref, "planes")


# ------------------------------------------------------------------------------------------------------------------
# wow_batch / wow_stream against single calls
# ------------------------------------------------------------------------------------------------------------------
BATCH_KW = [{"denoise_coefficients": [5, 2]}, {"bilateral": 1, "denoise_coefficients": [5, 2]},
            {"denoise_coefficients": [4, 1], "soft_threshold": False, "whitening": False, "weights": [0.5, 2]}]


def _stack(n, shape=(192, 256), dt=np.float32):
    return np.stack([_frame(shape, dt, seed=s) for s in range(n)])


@pytest.mark.parametrize("kw", range(len(BATCH_KW)))
def test_wow_batch_noise_forms_equal_single_calls(kw):
    import wavelets_b200 as wb
    kw = BATCH_KW[kw]
    frames = _stack(3)
    maps = np.stack([_photon_map(f) for f in frames])
    vec = np.array([0.5, 1.0, 2.0])
    forms = [("vec", vec, lambda i: float(vec[i])),
             ("vec_t", torch.from_numpy(vec).cuda(), lambda i: float(vec[i])),
             ("shared", maps[0], lambda i: maps[0]),
             ("per_frame", torch.from_numpy(maps), lambda i: maps[i])]
    for name, noise, single in forms:
        recon, planes, used = wb.wow_batch(frames, noise=noise, **kw)
        for i in range(len(frames)):
            r, co = wb.wow(frames[i], noise=single(i), **kw)
            r = torch.from_numpy(r).cuda()
            _assert_bitwise(recon[i], r, (name, i, "recon"))
            _assert_bitwise(planes[i], co.data, (name, i, "planes"))
        if name.startswith("vec"):
            assert used.dtype == torch.float64 and used.shape == (3,)
        else:
            assert used.dtype == torch.float32 and tuple(used.shape) == np.shape(noise)


def test_wow_batch_rejects_bad_noise_shapes():
    import wavelets_b200 as wb
    frames = _stack(3, shape=(64, 96))
    for bad in (np.ones(2), np.ones((64,)), np.ones((96,)), np.ones((2, 64, 96)), np.ones((64, 95)),
                np.ones((3, 1, 64, 96))):
        with pytest.raises(ValueError, match=r"\(B, H, W\)"):
            wb.wow_batch(frames, noise=bad, denoise_coefficients=[3])
        with pytest.raises(ValueError, match=r"\(B, H, W\)"):
            wb.wow_stream(frames, noise=bad, denoise_coefficients=[3])


@pytest.mark.parametrize("depth", [1, 2, 3])
def test_wow_stream_noise_forms_equal_single_calls(depth):
    import wavelets_b200 as wb
    frames = _stack(4)
    maps = np.stack([_photon_map(f) for f in frames])
    vec = np.array([0.5, 1.0, 2.0, 0.25])
    forms = [("vec", vec, lambda i: float(vec[i])), ("shared", maps[1], lambda i: maps[1]),
             ("per_frame", maps, lambda i: maps[i]),
             ("per_frame_pinned", torch.from_numpy(maps).pin_memory(), lambda i: maps[i])]
    for kw in BATCH_KW:
        for name, noise, single in forms:
            for inp in (frames, torch.from_numpy(frames).pin_memory()):
                out = wb.wow_stream(inp, depth=depth, noise=noise, **kw)
                out = out if isinstance(out, np.ndarray) else out.numpy()
                for i in range(len(frames)):
                    r, _ = wb.wow(frames[i], noise=single(i), **kw)
                    assert np.array_equal(out[i].view(np.int32), r.view(np.int32)), (name, kw, depth, i)
    # h > 0 takes wow() per frame, with each frame's map
    out = wb.wow_stream(frames, depth=depth, noise=maps, h=0.5, denoise_coefficients=[3, 1])
    for i in range(len(frames)):
        r, _ = wb.wow(frames[i], noise=maps[i], h=0.5, denoise_coefficients=[3, 1])
        assert np.array_equal(out[i], r), i


# ------------------------------------------------------------------------------------------------------------------
# Oracle parity and broadcasting
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dt", [np.float32, np.float64])
@pytest.mark.parametrize("kw", [{"denoise_coefficients": [5, 2]}, {"denoise_coefficients": [4, 2], "bilateral": 1},
                                {"denoise_coefficients": [4, 2], "soft_threshold": False}])
def test_wow_photon_map_oracle_parity(dt, kw):
    import wavelets_b200 as wb
    frame = orc.solar_like(256, seed=9, flux=0.05, dtype=dt)
    nmap = _photon_map(frame)
    recon, co = wb.wow(frame, noise=nmap, **kw)
    ref64, planes64, _ = orc.wow(frame.astype(np.float64), name="b3spline", backend="numpy",
                                 noise=nmap.astype(np.float64), **kw)
    # the thresholds bite: some but not all soft weights of scale 0 are below one half
    raw = orc.atrous_transform(frame.astype(np.float64), 2, "b3spline", bilateral=kw.get("bilateral"), backend="numpy")
    sig = orc.significance(raw, "b3spline", kw["denoise_coefficients"][0], 0, nmap.astype(np.float64),
                           bilateral=kw.get("bilateral"))
    frac = float((np.asarray(sig, dtype=np.float64) < 0.5).mean())
    assert 0.0 < frac < 1.0, frac
    if not kw.get("soft_threshold", True):
        # hard masks flip where |w| sits within rounding of the threshold: compare where the masks agree
        frac_off = (np.abs(recon - ref64) > 1e-4 * np.abs(ref64).max()).mean()
        assert frac_off < (5e-3 if dt == np.float32 else 1e-9), frac_off
        return
    if dt == np.float64:
        assert orc.emax(recon, ref64) <= 1e-12
        tol_p = 1e-12
    else:
        ref32, _, _ = orc.wow(frame, name="b3spline", backend="numpy", noise=nmap, **kw)
        assert orc.emax(recon, ref64) <= max(1e-5, 2 * orc.emax(ref32, ref64))
        tol_p = None
    if tol_p is not None:
        got = co.data.cpu().numpy()
        for p in range(len(planes64)):
            assert orc.emax(got[p], planes64[p]) <= (1e-11 if "bilateral" in kw else tol_p), p


def test_broadcast_maps():
    import wavelets_b200 as wb
    frame = orc.solar_like(128, seed=4, flux=0.05, dtype=np.float32)[:, :96].copy()
    row = (np.linspace(1, 3, 96)).astype(np.float32)
    col = (np.linspace(0.5, 2, 128)).astype(np.float32)[:, None]
    for m in (row, col):
        full = np.ascontiguousarray(np.broadcast_to(m, frame.shape))
        r_b, c_b = wb.wow(frame, noise=m, denoise_coefficients=[4, 2])
        r_f, c_f = wb.wow(frame, noise=full, denoise_coefficients=[4, 2])
        assert np.array_equal(r_b, r_f) and torch.equal(c_b.data, c_f.data)
        # Coefficients.significance / denoise / wow(Coefficients) broadcast the same way
        co_b = wb.AtrousTransform()(frame, 3)
        co_f = wb.AtrousTransform()(frame, 3)
        co_b.noise, co_f.noise = m, full
        assert torch.equal(co_b.significance(4, 0), co_f.significance(4, 0))
        co_b.denoise([4, 2])
        co_f.denoise([4, 2])
        assert torch.equal(co_b.data, co_f.data)
        co_b.noise = torch.from_numpy(m).cuda()
        co_f.noise = torch.from_numpy(full).cuda()
        r1, _ = wb.wow(co_b, denoise_coefficients=[4, 2])
        r2, _ = wb.wow(co_f, denoise_coefficients=[4, 2])
        assert torch.equal(r1, r2)
    for bad in (np.ones(95, np.float32), np.ones((127, 1), np.float32), np.ones((2, 128, 96), np.float32)):
        with pytest.raises(ValueError, match="broadcast"):
            wb.wow(frame, noise=bad, denoise_coefficients=[4])
        co = wb.AtrousTransform()(frame, 2)
        co.noise = bad
        with pytest.raises(ValueError, match="broadcast"):
            co.significance(4, 0)
