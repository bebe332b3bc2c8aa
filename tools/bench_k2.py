"""Timing of the two fp32 bilateral scale kernels, per scale (needs a CUDA device).

    python tools/bench_k2.py [--side 4096] [--reps 20] [--scales 0,1,3,6,9] [--out FILE.json]

Each scale is timed in the two call forms of atrous_scale(..., var_factor=1.0) that reach the two kernels:
"both" (c_{s+1} and w_s; the lean kernel, or the register-window kernel where the lean kernel declines the shape:
staged rows over 16 KiB, at the deepest dilations of rows wider than 4096 columns) and "c_only" (out_w=False; the
register-window kernel).  Also checks that the two give bit-identical c_{s+1}.  Only the public call is used, so the
script times any version of the library."""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import wavelets_b200 as wb  # noqa: E402
from wavelets_b200.wavelets import atrous_scale  # noqa: E402
from tools.bench_wow import solar_like_device, timed  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--side", type=int, default=4096)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--scales", default="0,1,3,6,9")
    ap.add_argument("--out", default=None, help="also write the results as JSON to this file")
    args = ap.parse_args()
    n = args.side
    img = solar_like_device(n, torch.float32).unsqueeze(0)
    res = {"side": n, "device": torch.cuda.get_device_name(0), "us": {}, "bit_identical": True}
    for sfc in (wb.B3spline, wb.Triangle):
        sf = sfc(2)
        for s in [int(x) for x in args.scales.split(",")]:
            c, w, c1 = torch.empty_like(img), torch.empty_like(img), torch.empty_like(img)
            row = {"both": 1e3 * timed(lambda: atrous_scale(img, s, sf, out_c=c, out_w=w, var_factor=1.0), args.reps),
                   "c_only": 1e3 * timed(lambda: atrous_scale(img, s, sf, out_c=c1, out_w=False, var_factor=1.0),
                                         args.reps)}
            same = torch.equal(c, c1)
            res["bit_identical"] &= same
            res["us"][f"{sf.name}_scale{s}"] = row
            print(sf.name, s, {k: round(v, 1) for k, v in row.items()}, "bit-identical" if same else "DIFFERENT",
                  flush=True)
    if args.out is None:
        return
    os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
