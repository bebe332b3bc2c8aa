"""GPU parity of denoise / significance / bilateral cascade / WOW / noise weights against the golden vectors of the
real reference and against the oracle evaluated in float64 (dual-oracle protocol of SURVEY.md 8(d))."""
import warnings

import numpy as np
import pytest
import torch

from oracle import atrous_oracle as orc
from tests.conftest import load_golden

pytestmark = pytest.mark.gpu


def _sf(name):
    import wavelets_b200 as wb
    return {"b3spline": wb.B3spline, "triangle": wb.Triangle}[name]


def dual_tol(ref_native, ref64, dt, fp64_tol=1e-12, base=1e-5):
    """fp64: fixed tolerance.  fp32: max(1e-5, 2 x the reference's own fp32-vs-fp64 distance) -- where the reference's
    fp32 path is itself further than 1e-5 from its fp64 path it cannot pin 1e-5 (SURVEY.md 8(d), Appendix C)."""
    if dt == "float64":
        return fp64_tol
    return max(base, 2 * orc.emax(ref_native, ref64))


def test_cfg1_readme_denoise_and_equivalences():
    """BASELINE configs[0] / README.md:37-61: Triangle, 512x512 np.random.normal, denoise([5, 3])."""
    import wavelets_b200 as wb
    g = load_golden("cfg1_denoise_triangle_512")
    np.random.seed(int(g["seed"]))
    img = np.random.normal(size=(512, 512))
    co = wb.AtrousTransform(wb.Triangle)(img, 2)
    assert orc.emax(co.data.cpu().numpy()[:, ::4, ::4], g["raw_sub"]) < 1e-13
    hard = co.significance(3, 1, soft_threshold=False)
    assert hard.dtype == torch.bool and int(hard.sum()) == int(g["hard_count"])
    assert np.array_equal(hard.cpu().numpy()[::4, ::4], g["hard_sub"])
    assert abs(co.noise - float(g["noise"])) <= 1e-15 * float(g["noise"])
    assert co.get_noise() == co.noise
    assert co.denoise([5, 3]) is None
    a = np.sum(co, axis=0)                       # README: coefficients accept numpy operations
    b = co.data.sum(axis=0).cpu().numpy()        # README: equivalent to coefficients.data.sum(axis=0)
    c = wb.denoise(img, [5, 3], wb.Triangle)     # README: the convenience function
    assert isinstance(c, np.ndarray) and c.dtype == np.float64
    assert np.array_equal(a, c) and orc.emax(b, c) < 1e-15
    assert orc.emax(c[::4, ::4], g["out_sub"]) < 1e-12
    assert abs(c.sum() - float(g["out_sum"])) < 1e-7


@pytest.mark.parametrize("dt", ["float32", "float64"])
def test_denoise_and_significance_golden(dt):
    import wavelets_b200 as wb
    g = load_golden(f"denoise_{dt}")
    img = g["img"]
    img64 = img.astype(np.float64)
    for sf in ("b3spline", "triangle"):
        co = wb.AtrousTransform(_sf(sf))(img, 3)
        noise = co.get_noise()
        assert isinstance(noise, np.float64)
        assert abs(noise - float(g[f"{sf}_noise"])) <= (3e-6 if dt == "float32" else 1e-13) * noise
        soft = co.significance(2.5, 2)
        assert soft.dtype == torch.float64
        assert np.abs(soft.cpu().numpy() - g[f"{sf}_soft2"]).max() < (2e-4 if dt == "float32" else 1e-11)
        hard = co.significance(3, 0, soft_threshold=False).cpu().numpy()
        assert hard.dtype == np.bool_ and (hard != g[f"{sf}_hard0"]).mean() < (1e-3 if dt == "float32" else 1e-9 + 0)
        assert torch.equal(co.significance(0, 1), torch.ones_like(co.data[0]))
        for key, kw in (("den_soft", dict(weights=[5, 3, 2])),
                        ("den_hard", dict(weights=[4, 3, 0], soft_threshold=False)),
                        ("den_noise", dict(weights=[3, 2], noise=0.8)),
                        ("den_bilateral", dict(weights=[3, 2], bilateral=1))):
            out = wb.denoise(img, scaling_function=_sf(sf), **kw)
            ref = g[f"{sf}_{key}"]
            assert out.dtype == ref.dtype and out.shape == ref.shape
            ref64 = orc.denoise(img64, name=sf, backend="numpy", **kw)
            if key == "den_hard":
                # a 1-ulp difference in w_s may flip a pixel that sits on the threshold
                frac = (np.abs(out - ref) > 1e-5 * np.abs(ref).max()).mean()
                assert frac < (2e-3 if dt == "float32" else 1e-9), (sf, key, frac)
            else:
                tol = dual_tol(ref, ref64, dt, fp64_tol=1e-11 if "bilateral" in key else 1e-12)
                assert orc.emax(out, ref64) <= tol, (sf, key, orc.emax(out, ref64), tol)


@pytest.mark.parametrize("dt", ["float32", "float64"])
def test_hard_mask_bit_exact_on_identical_planes(dt):
    """Identical plane values + explicit noise -> the hard significance mask is bit-exact (north_star)."""
    import wavelets_b200 as wb
    rng = np.random.default_rng(4)
    planes = rng.standard_normal((4, 200, 300)).astype(dt)
    for sf in ("b3spline", "triangle"):
        co = wb.Coefficients(torch.from_numpy(planes).cuda(), _sf(sf)(2))
        for noise in (0.731, np.float64(1.2345678901234), 0):
            co.noise = noise
            for s, sigma in ((0, 3), (1, 2.5), (2, 0.1)):
                want = orc.significance(planes, sf, sigma, s, noise, soft_threshold=False)
                got = co.significance(sigma, s, soft_threshold=False).cpu().numpy()
                assert np.array_equal(got.astype(want.dtype), want), (sf, noise, s)
        # noise=None: MAD estimate from the device median must reproduce np.median bit for bit
        co.noise = None
        want_noise = orc.get_noise(planes, sf)
        got = co.significance(3, 1, soft_threshold=False).cpu().numpy()
        assert co.noise == want_noise
        assert np.array_equal(got, orc.significance(planes, sf, 3, 1, want_noise, soft_threshold=False))
        # per-pixel noise map (watroo/wavelets.py:133)
        nmap = (0.5 + rng.uniform(size=(200, 300))).astype(dt)
        co.noise = nmap
        want = orc.significance(planes, sf, 2, 1, nmap, soft_threshold=False)
        assert np.array_equal(co.significance(2, 1, soft_threshold=False).cpu().numpy(), want)
        wsoft = orc.significance(planes, sf, 2, 1, nmap)
        assert np.abs(co.significance(2, 1).cpu().numpy() - wsoft).max() < 1e-12


@pytest.mark.parametrize("dt", ["float32", "float64"])
def test_bilateral_transform_golden(dt):
    import wavelets_b200 as wb
    g = load_golden(f"bilateral_{dt}")
    cases = [("in_solar", "solar_b1", "b3spline", 4, dict(bilateral=1)),
             ("in_solar", "solar_tri_b2", "triangle", 3, dict(bilateral=2.0)),
             ("in_gauss", "gauss_list_scaling", "b3spline", 4, dict(bilateral=[2, 1.5], bilateral_scaling=True))]
    for src, key, sf, level, kw in cases:
        img = g[src]
        co = wb.AtrousTransform(_sf(sf), **kw)(img, level)
        out = co.data.cpu().numpy()
        ref = g[key]
        assert out.dtype == ref.dtype and out.shape == ref.shape
        ref64 = orc.atrous_transform(img.astype(np.float64), level, sf, backend="numpy", **kw)
        for p in range(len(ref)):
            tol = dual_tol(ref[p], ref64[p], dt, fp64_tol=1e-11)
            floor = 4 * np.finfo(ref.dtype).eps * np.abs(img).max() / max(np.abs(ref64[p]).max(), 1e-300)
            assert orc.emax(out[p], ref64[p]) <= max(tol, floor), (key, p, orc.emax(out[p], ref64[p]), tol)


WOW_CASES = {
    "default": {},
    "den": dict(denoise_coefficients=[5, 2]),
    "den_hard": dict(denoise_coefficients=[5, 2], soft_threshold=False),
    "bil": dict(bilateral=1),
    "bil_den": dict(bilateral=1, denoise_coefficients=[5, 2]),
    "weights": dict(weights=[0.5, 2.0, 1.5], n_scales=3),
    "nowhite": dict(whitening=False, denoise_coefficients=[3, 1], noise=1.3),
    "tri": dict(scaling_function="triangle", denoise_coefficients=[0, 3]),
}


@pytest.mark.parametrize("dt", ["float32", "float64"])
def test_wow_golden(dt):
    import wavelets_b200 as wb
    g = load_golden(f"wow_{dt}")
    report = []
    for tag in ("gauss", "solar", "rect"):
        img = g[f"{tag}_in"]
        img64 = img.astype(np.float64)
        for key, kw in WOW_CASES.items():
            if f"{tag}_{key}_recon" not in g:
                continue
            kw = dict(kw)
            okw = dict(kw)
            sfname = kw.pop("scaling_function", "b3spline")
            okw.pop("scaling_function", None)
            keep = img.copy()
            recon, co = wb.wow(img, scaling_function=_sf(sfname), **kw)
            assert np.array_equal(img, keep)
            ref = g[f"{tag}_{key}_recon"]
            assert isinstance(recon, np.ndarray) and recon.dtype == ref.dtype and recon.shape == ref.shape
            assert isinstance(co, wb.Coefficients)
            ref64, planes64, noise64 = orc.wow(img64, name=sfname, backend="numpy", **okw)
            bil = "bil" in key
            ref_noise = float(g[f"{tag}_{key}_noise"])
            if np.isnan(ref_noise):
                assert co.noise is None
            else:
                assert abs(co.noise - ref_noise) <= (2e-4 if dt == "float32" else 1e-11) * abs(ref_noise)
            if key == "den_hard":
                frac = (np.abs(recon - ref64) > 1e-4 * np.abs(ref64).max()).mean()
                assert frac < (5e-3 if dt == "float32" else 1e-9), (tag, key, frac)
                continue
            tol = dual_tol(ref, ref64, dt, fp64_tol=1e-12)  # measured (float64): <= 1.1e-15 plain, <= 1.7e-14 bilateral
            e = orc.emax(recon, ref64)
            report.append((tag, key, e, tol))
            assert e <= tol, (tag, key, e, tol)
            if f"{tag}_{key}_planes" in g:
                rp = g[f"{tag}_{key}_planes"]
                got = co.data.cpu().numpy()
                assert got.shape == rp.shape and got.dtype == rp.dtype
                for p in range(len(rp)):
                    tp = dual_tol(rp[p], planes64[p], dt, fp64_tol=1e-11 if bil else 1e-12, base=2e-5)
                    assert orc.emax(got[p], planes64[p]) <= tp, (tag, key, p, orc.emax(got[p], planes64[p]), tp)
    print("\nwow parity (E_max vs float64 oracle, tolerance):")
    for row in report:
        print("  %-6s %-8s %.3e  (tol %.1e)" % row)


def test_wow_api_behaviour():
    """The reference's own test (tests/test_utils.py:7-9) plus the documented call surface."""
    import wavelets_b200 as wb
    ones = np.ones((128, 128))
    wowed, _ = wb.wow(ones)
    wowed, co = wb.wow(ones, bilateral=True)
    assert wowed.shape == (128, 128) and len(co) == wb.utils._wow_plan((128, 128), wb.B3spline, None, [], [], True)[0] + 1
    with pytest.raises(ValueError, match="Unknown input type"):
        wb.wow([[1.0, 2.0]])
    img = orc.solar_like(256, seed=5, flux=0.05, dtype=np.float32)
    # torch in -> torch out, coefficients whitened in place when passed back in
    t = torch.from_numpy(img).cuda()
    recon_t, co_t = wb.wow(t, denoise_coefficients=[5, 2])
    assert isinstance(recon_t, torch.Tensor) and recon_t.is_cuda
    recon_n, _ = wb.wow(img, denoise_coefficients=[5, 2])
    assert np.array_equal(recon_t.cpu().numpy(), recon_n)
    co_raw = wb.AtrousTransform(wb.B3spline)(img, len(co_t) - 1)
    recon_c, co_back = wb.wow(co_raw, denoise_coefficients=[5, 2])
    assert co_back is co_raw
    assert orc.emax(recon_c.cpu().numpy(), recon_n) < 1e-6
    assert orc.emax(co_raw.data.cpu().numpy(), co_t.data.cpu().numpy()) < 1e-6
    with warnings.catch_warnings(record=True) as rec:
        warnings.simplefilter("always")
        wb.wow(img[:64, :64], denoise_coefficients=[0] * 11, noise=1.0)
    assert any("lager" in str(w.message) for w in rec)
    # noise map route
    nmap = np.full(img.shape, 2.0, dtype=np.float32)
    r_map, _ = wb.wow(img, denoise_coefficients=[5, 2], noise=nmap)
    r_scalar, _ = wb.wow(img, denoise_coefficients=[5, 2], noise=2.0)
    assert orc.emax(r_map, r_scalar) < 1e-5


def test_wow_batch_matches_single_frames():
    import wavelets_b200 as wb
    frames = np.stack([orc.solar_like(256, seed=s, flux=0.05, dtype=np.float32) for s in (1, 2, 3)])
    recon, planes, noise = wb.wow_batch(frames, denoise_coefficients=[5, 2])
    assert recon.shape == (3, 256, 256) and planes.shape[0] == 3 and noise.shape == (3,)
    for b in range(3):
        r, co = wb.wow(frames[b], denoise_coefficients=[5, 2])
        assert np.array_equal(recon[b].cpu().numpy(), r)
        assert torch.equal(planes[b], co.data)
        assert noise[b].item() == co.noise
    rb, pb, _ = wb.wow_batch(frames[:2], bilateral=1)
    r0, c0 = wb.wow(frames[0], bilateral=1)
    assert np.array_equal(rb[0].cpu().numpy(), r0)


def _wow_per_scale(stack, scaling_function=None, n_scales=None, weights=(), denoise_coefficients=(), noise=None,
                   bilateral=None, bilateral_scaling=False, soft_threshold=True):
    """Reference for wb_wow_cascade: the same launches, issued one per-scale entry point at a time.  Per scale the fused
    wb_wow_scale, or where the scale is bilateral, the noise is a map, the MAD noise must first be estimated from the raw
    w_0 or the fused kernel declines: wb_atrous_scale[_bilateral] (+ wb_abs_median of the raw w_0) and the whitening K3.
    The noise is estimated lazily from the whitened plane 0 when the first threshold comes later.  Then the residual
    rescale and the synthesis.  ``stack`` is (B, H, W) on the device; returns (recon, planes, noise as a _Noise)."""
    import wavelets_b200 as wb
    from wavelets_b200 import _lib, utils
    from wavelets_b200.wavelets import _Noise, abs_median_noise, atrous_scale, plane_moments, synthesis
    lib = _lib.load(require_cuda=True)
    sfc = scaling_function or wb.B3spline
    b, h, w = stack.shape
    L, sigma_bilateral, wts, dns = utils._wow_plan((h, w), sfc, n_scales, weights, denoise_coefficients, bilateral)
    sf = sfc(2)
    sigma_e = sf.sigma_e(bilateral=sigma_bilateral)
    factors = [None] * L if sigma_bilateral is None else \
        wb.AtrousTransform(sfc, bilateral=sigma_bilateral, bilateral_scaling=bilateral_scaling).var_factors(L)
    nz = utils._stack_noise(noise, b, h, w, stack.dtype, stack.device)
    nz_map = None if nz is None else nz.map
    planes = torch.empty((b, L + 1, h, w), dtype=stack.dtype, device=stack.device)
    scratch = torch.empty((2, b, h, w), dtype=stack.dtype, device=stack.device)
    raw = torch.empty_like(stack)
    src = stack
    for s in range(L):
        dst_c = planes[:, L] if s == L - 1 else scratch[s & 1]
        d, wt = dns[s], wts[s]
        need_sig = d != 0
        mode = (1 if soft_threshold else 2) if need_sig else 0
        se = sigma_e[s] if need_sig else 1.0
        if need_sig and nz is None and s > 0:
            nz = _Noise(dev=abs_median_noise(planes[:, 0], sigma_e[0]))
        fused = factors[s] is None and nz_map is None and not (need_sig and nz is None) and \
            utils._wow_scale_fused(lib, src, dst_c, planes[:, s], s, sf, mode, d, se, nz if need_sig else _Noise(), wt)
        if not fused:
            atrous_scale(src, s, sf, out_c=dst_c, out_w=raw, var_factor=factors[s])
            if need_sig and nz is None:
                nz = _Noise(dev=abs_median_noise(raw, sigma_e[0]))
            if need_sig and nz_map is not None:
                utils._whiten_scale_map(lib, raw, planes[:, s], nz_map, s, sf, soft_threshold, d, sigma_e[s], wt)
            else:
                utils._whiten_scale(lib, raw, planes[:, s], s, sf, mode, d, se, nz if need_sig else _Noise(), wt)
        src = dst_c
    last = planes[:, L]
    mom = plane_moments(last)
    _lib.check(lib.wb_residual_rescale(last.data_ptr(), h * w, b, (L + 1) * h * w, _lib.dtype_code(stack.dtype),
                                       mom.data_ptr(), float(wts[L]), _lib.stream_ptr(stack.device)))
    return synthesis(planes), planes, nz


def test_wow_cascade_equals_per_scale_entry_points():
    """wb_wow_cascade (the whole WOW pipeline, plain or bilateral, in one library call) against the same launches issued
    per scale, bit for bit: default, MAD noise from the raw w_0 (scale 0) and from the whitened plane 0 (first threshold
    at scale 1), given noise (host scalar and device scalar), hard thresholds, weights, Triangle, float64, shapes the
    fused kernel declines (two-pass inside the call), batches."""
    import wavelets_b200 as wb
    cases = [((256, 256), np.float32, {}), ((256, 256), np.float32, {"denoise_coefficients": [5, 2]}),
             ((192, 320), np.float32, {"denoise_coefficients": [0, 3, 1]}),
             ((130, 1024), np.float32, {"denoise_coefficients": [4, 2], "noise": 0.7}),
             ((128, 2304), np.float32, {"denoise_coefficients": [4], "soft_threshold": False, "weights": [0.5, 2, 1.5]}),
             ((96, 201), np.float32, {"denoise_coefficients": [3, 1]}),                       # W % 4 != 0: generic kernels
             ((160, 160), np.float64, {"denoise_coefficients": [5, 2], "scaling_function": wb.Triangle}),
             ((64, 2560), np.float64, {"denoise_coefficients": [2]}),                         # fp64 beyond the fused kernel
             ((256, 256), np.float32, {"bilateral": 1, "denoise_coefficients": [5, 2]}),
             ((96, 1536), np.float32, {"bilateral": [1, 2], "denoise_coefficients": [0, 3], "bilateral_scaling": True}),
             ((128, 128), np.float64, {"bilateral": 1, "noise": 0.5, "denoise_coefficients": [4, 1]})]
    for shape, dt, kw in cases:
        img = orc.solar_like(max(shape), seed=3, flux=0.05, dtype=dt)[:shape[0], :shape[1]].copy()
        dev = torch.from_numpy(img).cuda()
        r1, c1 = wb.wow(dev, **kw)
        r0, p0, n0 = _wow_per_scale(dev.unsqueeze(0), **kw)
        assert torch.equal(r1, r0[0]) and torch.equal(c1.data, p0[0]), (shape, dt, kw)
        if n0 is None:
            assert c1.noise is None, (shape, kw)
        else:
            assert c1.noise == (n0.dev.item() if n0.dev is not None else n0.host), (shape, kw)
    dev_noise = torch.tensor([0.7], dtype=torch.float64, device="cuda")
    img = torch.from_numpy(orc.solar_like(256, seed=5, flux=0.05, dtype=np.float32)).cuda()
    r1, c1 = wb.wow(img, denoise_coefficients=[4, 2], noise=dev_noise)
    r0, p0, _ = _wow_per_scale(img.unsqueeze(0), denoise_coefficients=[4, 2], noise=dev_noise)
    assert torch.equal(r1, r0[0]) and torch.equal(c1.data, p0[0])
    nmap = torch.sqrt(1.5 * img.clamp(min=0) + 9)  # wb_wow_cascade_map
    for kw in ({"denoise_coefficients": [4, 0, 2]},
               {"bilateral": 1, "denoise_coefficients": [5, 2], "soft_threshold": False}):
        r1, c1 = wb.wow(img, noise=nmap, **kw)
        r0, p0, _ = _wow_per_scale(img.unsqueeze(0), noise=nmap, **kw)
        assert torch.equal(r1, r0[0]) and torch.equal(c1.data, p0[0]), kw
    frames = np.stack([orc.solar_like(256, seed=s, flux=0.05, dtype=np.float32) for s in (1, 2, 3)])
    rb1, pb1, nb1 = wb.wow_batch(frames, denoise_coefficients=[5, 2])
    rb0, pb0, nb0 = _wow_per_scale(torch.from_numpy(frames).cuda(), denoise_coefficients=[5, 2])
    assert torch.equal(rb1, rb0) and torch.equal(pb1, pb0) and torch.equal(nb1, nb0.dev)


def test_wow_stream_of_host_frames_matches_per_frame_calls():
    """wow_stream(): host frames in, host reconstructions out on three streams with one set of device buffers per frame
    in flight; every frame must equal wow(frame)[0] bit for bit, for the fused options (planned once), for the options
    that fall back to wow() per frame (h > 0), for NumPy and pinned inputs, and across repeated calls (buffer reuse)."""
    import wavelets_b200 as wb
    frames = np.stack([orc.solar_like(256, seed=s, flux=0.05, dtype=np.float32) for s in range(5)])
    for kw in ({}, {"denoise_coefficients": [5, 2]}, {"bilateral": 1, "denoise_coefficients": [5, 2]},
               {"weights": [0.5, 2], "whitening": False}, {"h": 0.5, "denoise_coefficients": [3, 1]}):
        out = wb.wow_stream(frames, **kw)
        assert isinstance(out, np.ndarray) and out.shape == frames.shape and out.dtype == np.float32
        for i in range(len(frames)):
            r, _ = wb.wow(frames[i], **kw)
            assert np.array_equal(out[i], r), (kw, i)
    pinned = torch.from_numpy(frames.astype(np.float64)).pin_memory()
    res = torch.empty_like(pinned).pin_memory()
    got = wb.wow_stream(pinned, out=res, depth=3, scaling_function=wb.Triangle, noise=0.01, denoise_coefficients=[4])
    assert got is res
    for i in range(len(frames)):
        r, _ = wb.wow(pinned[i].cuda(), scaling_function=wb.Triangle, noise=0.01, denoise_coefficients=[4])
        assert torch.equal(res[i], r.cpu())
    with pytest.raises(TypeError):
        wb.wow_stream(frames, no_such_option=1)
    with pytest.raises(ValueError):
        wb.wow_stream(frames[0])


@pytest.mark.parametrize("sf", ["b3spline", "triangle"])
def test_noise_weights(sf):
    import wavelets_b200 as wb
    g = load_golden(f"noise_weights_{sf}")
    out = _sf(sf)(2).compute_noise_weights(3, n_trials=2, fields=g["fields"])
    assert isinstance(out, np.ndarray) and out.dtype == np.float64 and out.shape == (3,)
    assert np.abs(out / g["out"] - 1).max() < 2e-6          # same fields as the reference run
    # device RNG path: statistical agreement with the recorded table (wavelets.py:245-247, :274-276)
    out2 = _sf(sf)(2).compute_noise_weights(6, n_trials=3, seed=11)
    table = _sf(sf)(2).sigma_e()[:6]
    assert np.abs(out2 / table - 1).max() < 0.03, out2 / table
    out3 = _sf(sf)(2).compute_noise_weights(6, n_trials=3, seed=11)
    assert np.array_equal(out2, out3)
    # 1-D signals and 3-D volumes (wavelets.py:225: side 11 * 2**n in every dimension) against their recorded tables;
    # the 1-D fields are short (11 * 2**n samples), hence the many trials and the looser bound
    w1 = _sf(sf)(1).compute_noise_weights(5, n_trials=400, seed=5)
    assert w1.shape == (5,) and np.abs(w1 / _sf(sf)(1).sigma_e()[:5] - 1).max() < 0.08, w1
    # (at side 88 the symmetric border weighs on scale 2: the oracle's own Monte-Carlo gives 0.935 x the table entry)
    w3 = _sf(sf)(3).compute_noise_weights(3, n_trials=2, seed=7)
    assert w3.shape == (3,) and np.abs(w3 / _sf(sf)(3).sigma_e()[:3] - 1).max() < 0.10, w3
    assert np.abs(w3[:2] / _sf(sf)(3).sigma_e()[:2] - 1).max() < 0.03, w3


@pytest.mark.parametrize("dt,bilateral", [(np.float32, None), (np.float32, 1), (np.float64, None)])
def test_wow_full_size_cfg3(dt, bilateral):
    """BASELINE cfg3 size: wow(4096^2 solar-like, [bilateral=1,] denoise_coefficients=[5, 2]).  Checks
    size-independent properties and an exact recomputation of sampled pixels of the whitening from the returned raw
    quantities."""
    import wavelets_b200 as wb
    n = 4096
    img = orc.solar_like(n, seed=2, flux=0.05, dtype=dt)
    dev = torch.from_numpy(img).cuda()
    recon, co = wb.wow(dev, bilateral=bilateral, denoise_coefficients=[5, 2])
    L = len(co) - 1
    assert L == 10 and co.data.shape == (11, n, n) and torch.isfinite(recon).all()
    # synthesis identity: recon == sum of the returned planes, in plane order
    acc = co.data[0].clone()
    for p in range(1, L + 1):
        acc += co.data[p]
    assert torch.equal(acc, recon)
    # residual plane has unit population std; whitened planes have local power ~ 1 where not thresholded
    assert abs(co.data[L].to(torch.float64).std(unbiased=False).item() - 1) < 1e-5
    # noise equals the MAD estimate of the raw first plane
    raw = wb.AtrousTransform(wb.B3spline, bilateral=None if bilateral is None else [bilateral] * (L + 1))(dev, L)
    want_noise = raw.get_noise()
    assert co.noise == want_noise
    # planes >= 2 carry no threshold: w' = w / sqrt(S[w^2]); verify on a strip against torch float64 arithmetic
    for s in (2, 5, 9):
        w = raw.data[s].to(torch.float64)
        power = wb.convolution((raw.data[s] ** 2), wb.B3spline(2), s=s).to(torch.float64)
        want = (w / torch.sqrt(torch.clamp(power, min=1e-15)))[1000:1016]
        got = co.data[s][1000:1016].to(torch.float64)
        assert ((got - want).abs().max() / want.abs().max()).item() < (2e-6 if dt == np.float32 else 1e-13)


@pytest.mark.parametrize("dt", ["float32", "float64"])
@pytest.mark.parametrize("sf", ["b3spline", "triangle"])
def test_wow_fused_scale_equals_two_pass(dt, sf):
    """wb_wow_scale (K1+K3 in one pass, raw w_s kept on chip) equals wb_atrous_scale followed by
    wb_wow_whiten_scale (bit for bit away from the top/bottom border), for every scale / significance mode / shape the fused kernel takes, and declines the rest."""
    import wavelets_b200 as wb
    from wavelets_b200 import _lib, utils
    from wavelets_b200.wavelets import atrous_scale
    lib = _lib.load(require_cuda=True)
    tdt = getattr(torch, dt)
    scf = _sf(sf)(2)
    gen = torch.Generator(device="cuda").manual_seed(7)
    # rows wider than 2048 fp32 columns take the lean packed kernel (wow_rows_lean_kernel), the others the generic one
    for (b, h, w) in ((1, 96, 128), (2, 67, 264), (1, 300, 1024), (1, 40, 2048), (3, 33, 32), (1, 70, 2304),
                      (2, 45, 4096), (1, 300, 3000)):
        src = torch.randn((b, h, w), generator=gen, device="cuda", dtype=tdt) * 3 + 1
        noise_dev = torch.tensor([0.7, 1.1, 0.9][:b], dtype=torch.float64, device="cuda")
        for s in range(0, 8):
            if (scf.taps_code // 2) * 2 ** s > w:
                break
            for mode, nz in ((0, utils._Noise()), (1, utils._Noise(dev=noise_dev)), (2, utils._Noise(host=0.8))):
                c_ref, w_raw = atrous_scale(src, s, scf)
                w_ref = torch.empty_like(src)
                utils._whiten_scale(lib, w_raw, w_ref, s, scf, mode, 2.5, 0.3, nz, 1.25)
                c_f, w_f = torch.full_like(src, float("nan")), torch.full_like(src, float("nan"))
                ok = utils._wow_scale_fused(lib, src, c_f, w_f, s, scf, mode, 2.5, 0.3, nz, 1.25)
                assert ok == bool(lib.wb_wow_scale_path(b, h, w, w, w, w, s, scf.taps_code, _lib.dtype_code(tdt),
                                                        src.data_ptr(), c_f.data_ptr(), w_f.data_ptr()))
                if w * src.element_size() > 16384:
                    assert not ok  # whole-row strips only: float64 rows wider than 2048 take the two-pass route
                    continue
                assert ok, (b, h, w, s)
                assert torch.equal(c_f, c_ref), (b, h, w, s, mode)
                # rows whose power window reaches beyond the top/bottom border see c_{s+1} of a virtual (reflected)
                # row, summed in the mirrored order: equal up to rounding there, bit-identical everywhere else
                edge = (scf.taps_code // 2) * 2 ** s
                if h > 2 * edge:
                    assert torch.equal(w_f[:, edge:h - edge], w_ref[:, edge:h - edge]), (b, h, w, s, mode)
                rel = (w_f - w_ref).abs() / w_ref.abs().max()
                tol = 1e-5 if dt == "float32" else 1e-13
                if mode == 2:  # an ulp in w_s may flip a coefficient that sits on the hard threshold
                    assert (rel > tol).float().mean().item() < 1e-3, (b, h, w, s, mode)
                else:
                    assert rel.max().item() < tol, (b, h, w, s, mode, rel.max().item())
    # shapes outside the fused kernel are declined before anything is launched
    wide = torch.randn((1, 16, 8192), device="cuda", dtype=tdt)
    out1, out2 = torch.zeros_like(wide), torch.zeros_like(wide)
    assert not utils._wow_scale_fused(lib, wide, out1, out2, 0, scf, 0, 0.0, 1.0, utils._Noise(), 1.0)
    odd = torch.randn((1, 16, 131), device="cuda", dtype=tdt)
    o1, o2 = torch.zeros_like(odd), torch.zeros_like(odd)
    assert not utils._wow_scale_fused(lib, odd, o1, o2, 0, scf, 0, 0.0, 1.0, utils._Noise(), 1.0)
    assert not out1.any() and not o1.any()
    # whole pipeline: wow() of the image (fused scales) and wow() of its coefficients (K3 on every raw plane) agree
    img = torch.from_numpy(orc.solar_like(512, seed=3, flux=0.05, dtype=np.dtype(dt).type)).cuda()
    for kw in ({}, dict(denoise_coefficients=[5, 2]), dict(denoise_coefficients=[0, 3], soft_threshold=False, noise=2.0),
               dict(weights=[0.5, 2.0], noise=1.5, denoise_coefficients=[4])):
        r1, c1 = wb.wow(img, scaling_function=_sf(sf), **kw)
        c2 = wb.AtrousTransform(_sf(sf))(img, len(c1) - 1)
        c2.noise = kw.get("noise")
        r2, _ = wb.wow(c2, **{k: v for k, v in kw.items() if k != "noise"})
        if kw.get("soft_threshold", True):
            assert orc.emax(r1.cpu().numpy(), r2.cpu().numpy()) < (1e-5 if dt == "float32" else 1e-12), kw
            assert orc.emax(c1.data.cpu().numpy(), c2.data.cpu().numpy()) < (1e-5 if dt == "float32" else 1e-12), kw
        else:
            rel = (c1.data - c2.data).abs() / c2.data.abs().amax(dim=(1, 2), keepdim=True)
            assert (rel > 1e-5).float().mean().item() < 1e-3, kw
        interior = slice(64, 512 - 64)  # scales 0-4 of the 512^2 frame: no virtual rows involved
        assert torch.equal(c1.data[:5, interior], c2.data[:5, interior]), kw


WOW_OPTION_CASES = {
    "gamma": dict(h=0.4, denoise_coefficients=[5, 2], gamma=2.5),
    "gamma_one": dict(h=1, denoise_coefficients=[3, 2, 1]),
    "gamma_range": dict(h=0.3, gamma_min=10.0, gamma_max=60.0, n_scales=3),
    "pv": dict(preserve_variance=True),
    "pv_den_gamma": dict(preserve_variance=True, h=0.25, denoise_coefficients=[4, 2], weights=[1.5, 0.5]),
}


@pytest.mark.parametrize("dt", ["float32", "float64"])
def test_wow_options_golden(dt):
    """SURVEY 8(f) rank 1: wow(h > 0) gamma blend and preserve_variance against the real reference's outputs and the
    float64 oracle (dual-oracle tolerance)."""
    import wavelets_b200 as wb
    g = load_golden(f"wow_options_{dt}")
    for tag in ("gauss", "solar"):
        img = g[f"{tag}_in"]
        img64 = img.astype(np.float64)
        for key, kw in WOW_OPTION_CASES.items():
            recon, co = wb.wow(img, **kw)
            ref, rp = g[f"{tag}_{key}_recon"], g[f"{tag}_{key}_planes"]
            assert isinstance(recon, np.ndarray) and recon.dtype == ref.dtype and recon.shape == ref.shape
            got = co.data.cpu().numpy()
            assert got.shape == rp.shape and got.dtype == rp.dtype
            ref64, planes64, _ = orc.wow(img64, backend="numpy", **kw)
            tol = dual_tol(ref, ref64, dt, fp64_tol=1e-12)
            assert orc.emax(recon, ref64) <= tol, (tag, key, orc.emax(recon, ref64), tol)
            for p in range(len(rp)):
                tp = dual_tol(rp[p], planes64[p], dt, fp64_tol=1e-12, base=2e-5)
                assert orc.emax(got[p], planes64[p]) <= tp, (tag, key, p, orc.emax(got[p], planes64[p]), tp)
    # Coefficients in -> whitened in place, same result as the image call
    img = g["solar_in"]
    r1, _ = wb.wow(img, h=0.4, denoise_coefficients=[5, 2], gamma=2.5)
    co = wb.AtrousTransform(wb.B3spline)(img, wb.utils._wow_plan(img.shape, wb.B3spline, None, [], [5, 2], None)[0])
    r2, co2 = wb.wow(co, h=0.4, denoise_coefficients=[5, 2], gamma=2.5)
    assert co2 is co and orc.emax(r2.cpu().numpy(), r1) < (1e-6 if dt == "float32" else 1e-13)


@pytest.mark.parametrize("dt", ["float32", "float64"])
def test_wow_nd_golden(dt):
    """wow() on 1-D signals and 3-D volumes (watroo/utils.py:121-219 is dimension-generic) against the real
    reference's outputs and the float64 oracle: default, thresholds + weights, gamma blend + preserve_variance, hard
    thresholds on a volume, bilateral volume."""
    import wavelets_b200 as wb
    from tests.test_oracle import WOW_ND_CASES
    g = load_golden(f"wow_nd_{dt}")
    for k, kw in enumerate(WOW_ND_CASES):
        kw = dict(kw)
        name = kw.pop("scaling_function", "b3spline")
        arr = g[f"in{k}"]
        keep = arr.copy()
        recon, co = wb.wow(arr, scaling_function=_sf(name), **kw)
        assert np.array_equal(arr, keep)
        ref_r, ref_p = g[f"recon{k}"], g[f"planes{k}"]
        assert isinstance(recon, np.ndarray) and recon.dtype == ref_r.dtype and recon.shape == ref_r.shape
        got = co.data.cpu().numpy()
        assert got.shape == ref_p.shape
        ref_noise = float(g[f"noise{k}"])
        if np.isnan(ref_noise):
            assert co.noise is None
        else:
            assert abs(co.noise / ref_noise - 1) < (2e-5 if dt == "float32" else 1e-12)
        r64, p64, _ = orc.wow(arr.astype(np.float64), name=name, backend="numpy", **kw)
        if not kw.get("soft_threshold", True):
            assert (np.abs(recon - r64) > 1e-4 * np.abs(r64).max()).mean() < (5e-3 if dt == "float32" else 1e-9)
            continue
        bil = "bilateral" in kw
        tol_r = dual_tol(ref_r, r64, dt, fp64_tol=1e-11 if bil else 1e-12)
        assert orc.emax(recon, r64) <= tol_r, (k, orc.emax(recon, r64), tol_r)
        for p in range(len(ref_p)):
            tp = dual_tol(ref_p[p], p64[p], dt, fp64_tol=1e-11 if bil else 1e-12, base=2e-5)
            assert orc.emax(got[p], p64[p]) <= tp, (k, p, orc.emax(got[p], p64[p]), tp)
