"""Parity at the widths the benchmark runs (VERDICT r1, "parity hole"): frames of 1536 .. 4096 columns, i.e. several
512-column strips of the bilateral kernels, the lean fused WOW kernel (rows wider than 2048 columns) and the lean K1.

Every comparison is CUDA path (through the C ABI) vs the float64 oracle on the same input, per plane, in the max norm
of SURVEY.md 8(d); the fp32 kernels are additionally reported against the reference's own fp32-vs-fp64 distance.  Each
test appends its measured E_max to gpurun_out/parity_report.txt (copied to profiles/ per round)."""
import os

import numpy as np
import pytest
import torch

from oracle import atrous_oracle as orc
from tests.conftest import ROOT, load_golden

pytestmark = pytest.mark.gpu

REPORT = os.path.join(ROOT, "gpurun_out", "parity_report.txt")


def report(line):
    print(line)
    try:
        os.makedirs(os.path.dirname(REPORT), exist_ok=True)
        with open(REPORT, "a") as fh:
            fh.write(line + "\n")
    except OSError:
        pass


def _sf(name):
    import wavelets_b200 as wb
    return {"b3spline": wb.B3spline, "triangle": wb.Triangle}[name]


def smooth_field(h, w, seed, dt):
    """Structured test frame: smooth large-scale gradients + Gaussian noise (positive, dynamic range ~50)."""
    rng = np.random.default_rng(seed)
    y, x = np.mgrid[0:h, 0:w]
    img = 40 + 25 * np.sin(x / 97.0) * np.cos(y / 31.0) + 10 * np.sin((x + 3 * y) / 11.0) + rng.standard_normal((h, w)) * 3
    return img.astype(dt)


# fp32 tolerances are the north-star 1e-5 per plane; the centred variance of K2 makes the fp32 kernel follow the float64
# oracle (the reference's own fp32 path is reported beside it).  fp64: 1e-12 (plain) and what exp() in double allows.
@pytest.mark.parametrize("dt", [np.float32, np.float64])
@pytest.mark.parametrize("sf", ["b3spline", "triangle"])
@pytest.mark.parametrize("shape", [(96, 4096), (40, 3000), (64, 1536), (33, 1032)])
def test_bilateral_scale_wide_vs_oracle(sf, dt, shape):
    """One bilateral scale (K2) on multi-strip rows, every dilation up to the single-reflection limit (d = 512 and 1024:
    the x halo is wider than a strip), both outputs, all pixels."""
    import wavelets_b200 as wb
    h, w = shape
    img = smooth_field(h, w, 3, dt)
    dev = torch.from_numpy(img).cuda()
    img64 = img.astype(np.float64)
    sfn = _sf(sf)(2)
    c = len(orc.TAPS[sf]) // 2
    worst_c = worst_w = 0.0
    for s in range(0, 12):
        if c * 2 ** s > w:
            break
        for vf in (1.0, 2.25 * (s + 1)):
            out_c, out_w = wb.atrous_scale(dev, s, sfn, var_factor=vf)
            var = orc.local_variance(img64, sf, s, backend="numpy") * vf
            ref_c = orc.bilateral_smooth(img64, sf, var, s)
            ref_w = img64 - ref_c
            ec, ew = orc.emax(out_c.cpu().numpy(), ref_c), orc.emax(out_w.cpu().numpy(), ref_w)
            worst_c, worst_w = max(worst_c, ec), max(worst_w, ew)
            tol_c, tol_w = (1e-6, 1e-5) if dt == np.float32 else (1e-13, 1e-11)
            assert ec <= tol_c and ew <= tol_w, (sf, shape, s, vf, ec, ew)
            # the two outputs are consistent: w = x - c exactly as stored
            assert torch.equal(out_w, dev - out_c)
    report(f"bilateral_scale {sf:8s} {np.dtype(dt).name} {h}x{w}: worst E_max c {worst_c:.2e}  w {worst_w:.2e}")


WIDE_WOW = {
    "default": {},
    "den": dict(denoise_coefficients=[5, 2]),
    "bil_den": dict(bilateral=1, denoise_coefficients=[5, 2]),
    "tri_bil": dict(scaling_function="triangle", bilateral=[1.5, 1], bilateral_scaling=True, denoise_coefficients=[0, 3]),
}


@pytest.mark.parametrize("dt", [np.float32, np.float64])
@pytest.mark.parametrize("shape,flux", [((512, 4096), 0.05), ((300, 2304), 0.01), ((200, 3000), 0.05)])
def test_wow_wide_vs_oracle(dt, shape, flux):
    """wow() on wide frames (lean fused kernel for fp32 W > 2048, multi-strip bilateral, two-pass fp64) against the
    float64 oracle: reconstruction and every whitened plane.  The dual-oracle floor E_max(ref32, ref64) is computed here
    with the oracle's native-dtype path and printed beside the measured error."""
    import wavelets_b200 as wb
    h, w = shape
    img = orc.solar_like(h, seed=7, flux=flux, dtype=dt, m=w)
    img64 = img.astype(np.float64)
    for key, kw in WIDE_WOW.items():
        kw = dict(kw)
        sfname = kw.pop("scaling_function", "b3spline")
        recon, co = wb.wow(img, scaling_function=_sf(sfname), **kw)
        got = co.data.cpu().numpy()
        ref64, planes64, noise64 = orc.wow(img64, name=sfname, backend="numpy", **kw)
        bil = "bilateral" in kw
        if dt == np.float32:
            ref32, planes32, _ = orc.wow(img, name=sfname, backend="numpy", **kw)
            floors = [orc.emax(planes32[p], planes64[p]) for p in range(len(planes64))]
            floor_r = orc.emax(ref32, ref64)
        else:
            floors, floor_r = [0.0] * len(planes64), 0.0
        if noise64 is not None:
            assert abs(co.noise - noise64) <= (3e-6 if dt == np.float32 else 1e-13) * abs(noise64), (key, co.noise, noise64)
        e_r = orc.emax(recon, ref64)
        errs = [orc.emax(got[p], planes64[p]) for p in range(len(planes64))]
        report(f"wow {key:8s} {np.dtype(dt).name} {h}x{w} L={len(errs) - 1}: recon {e_r:.2e} (ref32-vs-ref64 {floor_r:.2e}); "
               f"planes max {max(errs):.2e} (floor max {max(floors):.2e})")
        if dt == np.float32:
            # Whitened fp32 planes: both the reference's fp32 path and ours carry the rounding of the stored c_s (0.5 ulp
            # of values ~400 against details ~0.05 in quiet regions, amplified by 1 / sqrt(P)); ours adds the roundings
            # of the separable fp32 FMA chains (the reference's DFT branch rounds once).  Measured (r2, parity report):
            # <= 3.3e-5 where the reference's own fp32-vs-fp64 distance is 1.1e-5.
            assert e_r <= max(1e-5, 2 * floor_r), (key, e_r, floor_r)
            for p, (e, f) in enumerate(zip(errs, floors)):
                assert e <= max(2e-5, 4 * f), (key, p, e, f)
        else:
            tol = 1e-10 if bil else 1e-12
            assert e_r <= tol and max(errs) <= tol, (key, e_r, errs)


@pytest.mark.parametrize("dt", ["float32", "float64"])
def test_wide_golden_from_reference(dt):
    """Outputs of the REAL reference on 96x4096 and 72x1536 frames (tests/golden/make_golden.py --wide), stored on a
    column subset that brackets every 512-column strip boundary."""
    import wavelets_b200 as wb
    g = load_golden(f"wide_{dt}")
    npdt = np.dtype(dt).type
    for tag in ("a", "b"):
        h, w, seed = (int(v) for v in g[f"{tag}_shape"])
        img = orc.solar_like(h, seed=seed, flux=float(g[f"{tag}_flux"]), dtype=npdt, m=w)
        assert img.astype(np.float64).sum() == float(g[f"{tag}_in_sum"]) and np.array_equal(img[:2], g[f"{tag}_in_rows"])
        img64 = img.astype(np.float64)
        cols = g[f"{tag}_cols"]
        cases = [("plain", "b3spline", 5, {}), ("bil", "b3spline", 5, dict(bilateral=1)),
                 ("tri_bil", "triangle", 6, dict(bilateral=[1.5, 1], bilateral_scaling=True))]
        for key, sf, level, kw in cases:
            out = wb.AtrousTransform(_sf(sf), **kw)(img, level).data.cpu().numpy()[:, :, cols]
            ref = g[f"{tag}_{key}"]
            ref64 = orc.atrous_transform(img64, level, sf, backend="numpy", **kw)[:, :, cols]
            assert out.shape == ref.shape and out.dtype == ref.dtype
            for p in range(level + 1):
                floor = orc.emax(ref[p], ref64[p])
                e = orc.emax(out[p], ref64[p])
                # fp32 bilateral on flux=1 frames: the reference's own fp32 variance cancels catastrophically
                # (SURVEY Appendix C), so its fp32 planes sit far from its float64 planes; ours follow the float64 ones
                tol = max(1e-5, 2 * floor) if dt == "float32" else (1e-11 if kw else 1e-12)
                assert e <= tol, (tag, key, p, e, floor)
                if dt == "float64":
                    # against the reference's own float64 output: it sits `floor` away from the separable float64 sum
                    # (DFT rounding, 4e-11 on the flux = 1 frame), so that distance is all this comparison can pin
                    assert orc.emax(out[p], ref[p]) <= 2 * floor + (1e-11 if kw else 1e-12), (tag, key, p)
        for key, kw in (("default", {}), ("den", dict(denoise_coefficients=[5, 2])),
                        ("bil_den", dict(bilateral=1, denoise_coefficients=[5, 2]))):
            recon, co = wb.wow(img, **kw)
            ref_r, ref_p = g[f"{tag}_{key}_recon"], g[f"{tag}_{key}_planes"]
            r64, p64, n64 = orc.wow(img64, backend="numpy", **kw)
            got_p = co.data.cpu().numpy()[:, :, cols]
            assert recon.dtype == ref_r.dtype and got_p.shape == ref_p.shape
            ref_noise = float(g[f"{tag}_{key}_noise"])
            if not np.isnan(ref_noise):
                assert abs(co.noise - ref_noise) <= (2e-4 if dt == "float32" else 1e-11) * abs(ref_noise)
            bil = "bilateral" in kw
            floor = orc.emax(ref_r, r64[:, cols])
            e = orc.emax(recon[:, cols], r64[:, cols])
            report(f"wide golden {tag} {key:8s} {dt}: recon vs ref64 {e:.2e} (reference fp-native vs ref64 {floor:.2e})")
            assert e <= (max(1e-5, 2 * floor) if dt == "float32" else (1e-10 if bil else 1e-12)), (tag, key, e, floor)
            for p in range(len(ref_p)):
                fl = orc.emax(ref_p[p], p64[p][:, cols])
                ep = orc.emax(got_p[p], p64[p][:, cols])
                assert ep <= (max(2e-5, 4 * fl) if dt == "float32" else (1e-10 if bil else 1e-12)), (tag, key, p, ep, fl)
                if dt == "float64":
                    assert orc.emax(got_p[p], ref_p[p]) <= 2 * fl + (1e-10 if bil else 1e-12), (tag, key, p)


@pytest.mark.parametrize("dt", [np.float32, np.float64])
def test_lean_fused_wow_scale_vs_oracle(dt):
    """One fused WOW scale (wb_wow_scale: the lean kernel for fp32 rows wider than 2048 columns) directly against the
    oracle -- smooth, detail, local power and whitening in float64 -- for W in {2304, 4096}, every dilation."""
    import wavelets_b200 as wb
    from wavelets_b200 import _lib, utils
    lib = _lib.load(require_cuda=True)
    sfn = wb.B3spline(2)
    for (h, w) in ((80, 2304), (130, 4096), (44, 3000), (36, 3592)):
        if dt == np.float64 and w > 2048:
            w //= 2  # fp64 rows beyond 2048 columns are outside the fused kernel (two-pass route, tested above)
        img = smooth_field(h, w, 9, dt)
        dev = torch.from_numpy(img).cuda().unsqueeze(0)
        img64 = img.astype(np.float64)
        for s in range(0, 11):
            if 2 * 2 ** s > w:
                break
            c_f, w_f = torch.empty_like(dev), torch.empty_like(dev)
            assert utils._wow_scale_fused(lib, dev, c_f, w_f, s, sfn, 1, 2.0, 0.4, utils._Noise(host=0.9), 1.5)
            c64 = orc.smooth(img64, "b3spline", s, backend="numpy")
            w64 = img64 - c64
            p64 = orc.smooth(w64 ** 2, "b3spline", s, backend="numpy")
            p64[p64 <= 0] = 1e-15
            from scipy.special import erf
            want = w64 * erf(np.abs(w64 / (2.0 * 0.9 * 0.4))) * (1.5 / np.sqrt(p64))
            ec, ew = orc.emax(c_f[0].cpu().numpy(), c64), orc.emax(w_f[0].cpu().numpy(), want)
            assert ec <= (1e-6 if dt == np.float32 else 1e-14), (w, s, ec)
            assert ew <= (1e-5 if dt == np.float32 else 1e-12), (w, s, ew)
    report(f"lean fused wow scale {np.dtype(dt).name}: all dilations within tolerance")


@pytest.mark.parametrize("dt", [np.float32, np.float64])
@pytest.mark.parametrize("sf", ["b3spline", "triangle"])
def test_lean_k1_k3_every_dilation_vs_oracle(sf, dt):
    """The lean K1 (one cascade scale) and K3 (whitening of a raw detail plane) kernels on short frames of 1032 .. 11264
    columns at EVERY dilation the single-reflection limit allows: from d = 32 (fp32) / 16 (fp64) on a thread's two column
    vectors are one dilation step apart (paired columns), with partial pair blocks and masked second vectors at widths
    that are not a multiple of 2 d (3000, 3592, 1032), and mirrored taps on both sides at the deep scales; rows wider
    than one ring slot (8192, 11264 fp32; 2304 .. 4096 fp64) run as column strips with halo columns, the last strip
    partial."""
    import wavelets_b200 as wb
    from wavelets_b200 import _lib, utils
    from scipy.special import erf
    lib = _lib.load(require_cuda=True)
    sfn = _sf(sf)(2)
    c_taps = len(sfn.coefficients_1d) // 2
    f32 = dt == np.float32
    worst_c = worst_w = worst_k3 = 0.0
    shapes = ((40, 4096), (44, 3000), (36, 3592), (52, 2304), (33, 1032), (24, 8192), (20, 11264), (22, 6000))
    for (h, w) in shapes:
        if not f32 and w > 6000:
            continue
        img = smooth_field(h, w, 11 + w, dt)
        dev = torch.from_numpy(img).cuda()
        img64 = img.astype(np.float64)
        for s in range(0, 12):
            if c_taps * 2 ** s > w:
                break
            c1, w1 = wb.atrous_scale(dev, s, sfn)
            c64 = orc.smooth(img64, sf, s, backend="numpy")
            ec, ew = orc.emax(c1.cpu().numpy(), c64), orc.emax(w1.cpu().numpy(), img64 - c64)
            assert ec <= (1e-6 if f32 else 1e-14) and ew <= (5e-6 if f32 else 1e-13), (sf, w, s, ec, ew)
            # K3 on the raw plane this launch wrote: w' = w * erf(|w| / (sigma noise sigma_e)) * weight / sqrt(P)
            out = torch.empty_like(w1).unsqueeze(0)
            utils._whiten_scale(lib, w1.unsqueeze(0), out, s, sfn, 1, 2.0, 0.4, utils._Noise(host=0.9), 1.5)
            wr = w1.cpu().numpy().astype(np.float64)
            p64 = orc.smooth(wr ** 2, sf, s, backend="numpy")
            p64[p64 <= 0] = 1e-15
            want = wr * erf(np.abs(wr / (2.0 * 0.9 * 0.4))) * (1.5 / np.sqrt(p64))
            ek = orc.emax(out[0].cpu().numpy(), want)
            assert ek <= (1e-5 if f32 else 1e-12), (sf, w, s, ek)
            worst_c, worst_w, worst_k3 = max(worst_c, ec), max(worst_w, ew), max(worst_k3, ek)
    report(f"lean K1 / K3 {sf} {np.dtype(dt).name}, every dilation, W in 1032..11264: worst E_max c {worst_c:.2e}  "
           f"w {worst_w:.2e}  whitened {worst_k3:.2e}")


@pytest.mark.parametrize("sf", ["b3spline", "triangle"])
def test_bilateral_kernel_variants_bit_identical(sf):
    """The two fp32 K2 kernels perform the same operations in the same order: the lean kernel (the default call, both
    outputs) and the register-window kernel (one output: out_w=False or out_c=False) give bit-identical c_{s+1} and w_s
    on multi-strip frames, every dilation, batch of 2."""
    import wavelets_b200 as wb
    from torch.profiler import ProfilerActivity, profile
    sfn = _sf(sf)(2)
    c = len(orc.TAPS[sf]) // 2
    gen = torch.Generator(device="cuda").manual_seed(5)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for (b, h, w) in ((1, 70, 4096), (2, 33, 1032), (1, 257, 512)):
            src = torch.randn((b, h, w), generator=gen, device="cuda") * 3 + 20
            for s in range(0, 31):
                if c * 2 ** s > w:
                    break
                lean_c, lean_w = wb.atrous_scale(src, s, sfn, var_factor=1.7)
                window_c, _ = wb.atrous_scale(src, s, sfn, var_factor=1.7, out_w=False)
                _, window_w = wb.atrous_scale(src, s, sfn, var_factor=1.7, out_c=False)
                assert torch.equal(window_c, lean_c) and torch.equal(window_w, lean_w), (sf, b, h, w, s)
        torch.cuda.synchronize()
    # both kernels ran, so the comparison above is one between them
    names = {ev.name for ev in prof.events()}
    for kern in ("bilateral_lean_kernel", "bilateral_window_kernel"):
        assert any(kern in n for n in names), (kern, sorted(names))


@pytest.mark.parametrize("dt", [np.float32, np.float64])
def test_degenerate_thresholds_stay_finite(dt):
    """ADVICE r1: a denormal noise scalar (1 / threshold overflows in fp32) and a tiny bilateral variance factor must
    not poison pixels whose coefficient / tap difference is exactly zero (flat patches) -- the reference yields 0 / a
    weight of 1 there."""
    import wavelets_b200 as wb
    img = orc.solar_like(128, seed=8, flux=0.05, dtype=dt, m=256)
    img[32:96, 64:192] = 7.0  # flat patch: w_s == 0 exactly in its interior
    recon, co = wb.wow(img, denoise_coefficients=[5, 2], noise=1e-42)
    assert np.isfinite(recon).all() and torch.isfinite(co.data).all()
    ref, planes, _ = orc.wow(img.astype(np.float64), backend="numpy", denoise_coefficients=[5, 2], noise=1e-42)
    assert orc.emax(recon, ref) <= (1e-5 if dt == np.float32 else 1e-12)
    dev = torch.from_numpy(img).cuda()
    c, w = wb.atrous_scale(dev, 1, wb.B3spline(2), var_factor=1e-30)
    assert torch.isfinite(c).all() and torch.isfinite(w).all()
    assert torch.equal(c[50:70, 100:150], dev[50:70, 100:150])  # all taps equal: the smooth returns the pixel itself
