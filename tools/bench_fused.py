"""Per-scale launch time of the fused WOW scale kernel and of wow() itself (GPU box only).

    python tools/bench_fused.py [--side 4096] [--reps 30] [--tag name]
"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import wavelets_b200 as wb  # noqa: E402
from wavelets_b200 import _lib, utils  # noqa: E402
from tools.bench_wow import solar_like_device, timed  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--side", type=int, default=4096)
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--tag", default="")
    ap.add_argument("--dtype", default="f32")
    args = ap.parse_args()
    lib = _lib.load(require_cuda=True)
    n = args.side
    tdt = torch.float32 if args.dtype == "f32" else torch.float64
    img = solar_like_device(n, tdt)
    sf = wb.B3spline(2)
    src = img.unsqueeze(0)
    c = torch.empty_like(src)
    o = torch.empty_like(src)
    nz = utils._Noise(dev=torch.tensor([1.0], dtype=torch.float64, device="cuda"))
    res = {"tag": args.tag, "side": n, "dtype": args.dtype, "env": {k: v for k, v in os.environ.items() if k.startswith("WB_")}}
    fusable = bool(utils._wow_scale_fused(lib, src, c, o, 3, sf, 0, 0.0, 1.0, utils._Noise(), 1.0))
    if fusable:
        res["fused_us"] = [round(1e3 * timed(lambda: utils._wow_scale_fused(lib, src, c, o, s, sf, 0, 0.0, 1.0, utils._Noise(), 1.0),
                                             args.reps), 2) for s in range(10)]
        res["fused_soft_us"] = [round(1e3 * timed(lambda: utils._wow_scale_fused(lib, src, c, o, s, sf, 1, 5.0, 0.2, nz, 1.0),
                                                  args.reps), 2) for s in range(10)]
    from wavelets_b200.wavelets import atrous_scale
    w = torch.empty_like(src)
    res["k1_us"] = [round(1e3 * timed(lambda: atrous_scale(src, s, sf, out_c=c, out_w=w), args.reps), 2) for s in range(10)]
    res["k3_us"] = [round(1e3 * timed(lambda: utils._whiten_scale(lib, w, o, s, sf, 0, 0.0, 1.0, utils._Noise(), 1.0), args.reps), 2)
                    for s in range(10)]
    # kernel-switch cost: the same launches back to back, grouped by kernel (s4 x4, s5 x4) and alternating (s4, s5) x4
    def seq(order):
        for s in order:
            atrous_scale(src, s, sf, out_c=c, out_w=w)
    res["switch_us"] = {"grouped_4_5": round(1e3 * timed(lambda: seq([4] * 4 + [5] * 4), args.reps) / 8, 2),
                        "alternating_4_5": round(1e3 * timed(lambda: seq([4, 5] * 4), args.reps) / 8, 2),
                        "grouped_0_1_4_5": round(1e3 * timed(lambda: seq([0] * 2 + [1] * 2 + [4] * 2 + [5] * 2), args.reps) / 8, 2),
                        "alternating_0_1_4_5": round(1e3 * timed(lambda: seq([0, 1, 4, 5] * 2), args.reps) / 8, 2)}
    res["k3_soft_us"] = [round(1e3 * timed(lambda: utils._whiten_scale(lib, w, o, s, sf, 1, 5.0, 0.2, nz, 1.0), args.reps), 2)
                         for s in range(10)]

    def fseq(order):
        for s in order:
            utils._wow_scale_fused(lib, src, c, o, s, sf, 0, 0.0, 1.0, utils._Noise(), 1.0)
    res["switch_fused_us"] = {} if not fusable else {"grouped_0_1_4_5": round(1e3 * timed(lambda: fseq([0] * 2 + [1] * 2 + [4] * 2 + [5] * 2), args.reps) / 8, 2),
                              "alternating_0_1_4_5": round(1e3 * timed(lambda: fseq([0, 1, 4, 5] * 2), args.reps) / 8, 2),
                              "grouped_4_5": round(1e3 * timed(lambda: fseq([4] * 4 + [5] * 4), args.reps) / 8, 2),
                              "alternating_4_5": round(1e3 * timed(lambda: fseq([4, 5] * 4), args.reps) / 8, 2)}
    tr = wb.AtrousTransform(wb.B3spline)
    res["transform_ms"] = round(timed(lambda: tr(img, 10), 100), 4)
    res["wow_ms"] = round(timed(lambda: wb.wow(img), args.reps), 4)
    res["wow_den_ms"] = round(timed(lambda: wb.wow(img, denoise_coefficients=[5, 2], noise=1.0), args.reps), 4)
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
