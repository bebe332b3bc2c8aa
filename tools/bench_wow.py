"""Device-resident timing of the WOW variants and of every kernel family they are made of (GPU box only).

    python tools/bench_wow.py [--side 4096] [--dtype f32|f64] [--reps 20] [--out gpurun_out/bench_wow.json]

Reports 4096^2 WOW frames/s (default / denoise / bilateral+denoise, BASELINE.json configs[2]) with the algorithmic-byte
roofline of SURVEY.md 8(d) ((5L+3)*sizeof(T) per pixel), and microseconds per launch for each kernel per scale.
"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import wavelets_b200 as wb  # noqa: E402
from wavelets_b200 import _lib, utils  # noqa: E402
from wavelets_b200.wavelets import abs_median_noise, atrous_scale, plane_moments, synthesis  # noqa: E402


def timed(fn, reps, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps  # ms


def solar_like_device(n, dtype, seed=2):
    """Closed-form solar-like frame generated on the device (disk + corona + blobs + Poisson-like noise)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    y, x = torch.meshgrid(torch.arange(n, device="cuda", dtype=torch.float64),
                          torch.arange(n, device="cuda", dtype=torch.float64), indexing="ij")
    r = torch.hypot(x - n / 2, y - n / 2) / (0.4 * n)
    img = torch.where(r < 1, 2000 * (0.4 + 0.6 * torch.sqrt(torch.clamp(1 - r ** 2, min=0))),
                      800 * torch.exp(-(torch.clamp(r, min=1) - 1) / 0.15))
    for _ in range(30):
        cx, cy = (torch.rand(2, generator=g, device="cuda") * 0.6 + 0.2) * n
        sg = (torch.rand(1, generator=g, device="cuda") * 27 + 3) * n / 1024
        amp = torch.rand(1, generator=g, device="cuda") * 7500 + 500
        img += amp * torch.exp(-((x - cx) ** 2 + (y - cy) ** 2) / (2 * sg ** 2))
    img = (img + 20) * 0.05
    img = img + torch.sqrt(img) * torch.randn(img.shape, generator=g, device="cuda", dtype=torch.float64)
    return torch.round(torch.clamp(img, min=0)).to(dtype)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--side", type=int, default=4096)
    ap.add_argument("--dtype", default="f32")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default="gpurun_out/bench_wow.json")
    args = ap.parse_args()
    lib = _lib.load(require_cuda=True)
    tdt = torch.float32 if args.dtype == "f32" else torch.float64
    es = 4 if args.dtype == "f32" else 8
    n = args.side
    peak = 6530.0
    pk = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "MEASURED_PEAKS.json")
    if os.path.exists(pk):
        peak = float(json.load(open(pk))["hbm_gbs"])
    img = solar_like_device(n, tdt)
    sf = wb.B3spline(2)
    res = {"side": n, "dtype": args.dtype, "peak_gbs": peak, "wow": {}, "kernels": {}}

    for name, kw in (("default", {}), ("den", dict(denoise_coefficients=[5, 2])),
                     ("bil_den", dict(bilateral=1, denoise_coefficients=[5, 2])), ("bil", dict(bilateral=1))):
        ms = timed(lambda: wb.wow(img, **kw), args.reps)
        L = len(wb.wow(img, **kw)[1]) - 1
        algo = (5 * L + 3) * es * n * n
        res["wow"][name] = {"ms": ms, "frames_per_s": 1e3 / ms, "scales": L, "algorithmic_gb": algo / 1e9,
                            "achieved_gbs": algo / ms / 1e6, "frac": algo / ms / 1e6 / peak}
        print(name, f"{ms:.3f} ms  {1e3 / ms:.1f} frames/s  "
              f"{algo / ms / 1e6:.0f} GB/s algorithmic ({algo / ms / 1e6 / peak:.1%})", flush=True)

    # per-kernel, per-scale launch times (k1 + k3_whiten against fused: the two-pass and the fused route of a scale)
    src = img.unsqueeze(0)
    c = torch.empty_like(src)
    w = torch.empty_like(src)
    o = torch.empty_like(src)
    planes = torch.randn((11, n, n), device="cuda", dtype=tdt)
    nz = utils._Noise(dev=torch.tensor([1.0], dtype=torch.float64, device="cuda"))
    for s in range(10):
        row = {}
        row["k1_us"] = 1e3 * timed(lambda: atrous_scale(src, s, sf, out_c=c, out_w=w), args.reps)
        row["k2_bilateral_us"] = 1e3 * timed(lambda: atrous_scale(src, s, sf, out_c=c, out_w=w, var_factor=1.0), args.reps)
        row["k3_whiten_us"] = 1e3 * timed(lambda: utils._whiten_scale(lib, w, o, s, sf, 0, 0.0, 1.0, utils._Noise(), 1.0), args.reps)
        row["k3_whiten_soft_us"] = 1e3 * timed(lambda: utils._whiten_scale(lib, w, o, s, sf, 1, 5.0, 0.2, nz, 1.0), args.reps)
        row["fused_us"] = 1e3 * timed(lambda: utils._wow_scale_fused(lib, src, c, o, s, sf, 0, 0.0, 1.0, utils._Noise(), 1.0), args.reps)
        row["fused_soft_us"] = 1e3 * timed(lambda: utils._wow_scale_fused(lib, src, c, o, s, sf, 1, 5.0, 0.2, nz, 1.0), args.reps)
        res["kernels"][f"scale{s}"] = row
        print(s, {k: round(v, 1) for k, v in row.items()}, flush=True)
    res["kernels"]["abs_median_us"] = 1e3 * timed(lambda: abs_median_noise(w, 0.89), args.reps)
    res["kernels"]["plane_moments_us"] = 1e3 * timed(lambda: plane_moments(w), args.reps)
    res["kernels"]["synthesis11_us"] = 1e3 * timed(lambda: synthesis(planes), args.reps)
    print({k: v for k, v in res["kernels"].items() if not k.startswith("scale")})
    os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
