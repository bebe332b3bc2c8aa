"""K1 on rows wider than one ring slot (column strips): per-scale launch time and whole transforms (GPU box only).

    python tools/bench_wide.py [--tag name]
"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import wavelets_b200 as wb  # noqa: E402
from wavelets_b200.wavelets import atrous_scale  # noqa: E402
from tools.bench_wow import timed  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tag", default="")
    args = ap.parse_args()
    sf = wb.B3spline(2)
    res = {"tag": args.tag, "env": {k: v for k, v in os.environ.items() if k.startswith("WB_")}}
    for name, shape in (("band_4096x32768", (4096, 32768)), ("frame_8192", (8192, 8192))):
        src = torch.randn(shape, device="cuda")
        c, w = torch.empty_like(src), torch.empty_like(src)
        res[name + "_k1_us"] = [round(1e3 * timed(lambda: atrous_scale(src, s, sf, out_c=c, out_w=w), 10), 1) for s in range(11)]
        del c, w
        tr = wb.AtrousTransform(wb.B3spline)
        res[name + "_transform10_ms"] = round(timed(lambda: tr(src, 10), 5), 3)
        del src
        torch.cuda.empty_cache()
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
