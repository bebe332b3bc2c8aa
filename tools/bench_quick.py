"""Quick device-resident timings of the three headline calls (GPU box only), for A/B runs under environment switches
(WB_L2_HINTS, WB_PDL).

    python tools/bench_quick.py [--reps 200] [--tag name]"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import wavelets_b200 as wb  # noqa: E402
from tools.bench_wow import solar_like_device, timed  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--tag", default="")
    ap.add_argument("--side", type=int, default=4096)
    args = ap.parse_args()
    n = args.side
    img = torch.randn((n, n), device="cuda")
    solar = solar_like_device(n, torch.float32)
    tr = wb.AtrousTransform(wb.B3spline)
    res = {"tag": args.tag, "env": {k: v for k, v in os.environ.items() if k.startswith("WB_")}}
    res["transform_ms"] = timed(lambda: tr(img, 10), args.reps)
    res["transform_mpx_scales_per_s"] = n * n * 10 / res["transform_ms"] / 1e3
    res["wow_ms"] = timed(lambda: wb.wow(solar), max(10, args.reps // 4))
    res["wow_den_ms"] = timed(lambda: wb.wow(solar, denoise_coefficients=[5, 2]), max(10, args.reps // 4))
    res["wow_bilateral_ms"] = timed(lambda: wb.wow(solar, bilateral=1, denoise_coefficients=[5, 2]), max(5, args.reps // 10))
    s64 = solar.to(torch.float64)
    res["wow_f64_ms"] = timed(lambda: wb.wow(s64), 10)
    res["wow_bilateral_f64_ms"] = timed(lambda: wb.wow(s64, bilateral=1, denoise_coefficients=[5, 2]), 4)
    del s64
    stack = solar.unsqueeze(0).repeat(8, 1, 1)
    res["wow_batch8_ms_per_frame"] = timed(lambda: wb.wow_batch(stack), 5) / 8
    p = torch.cuda.get_device_properties(0)
    res["l2_bytes"] = p.L2_cache_size
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
