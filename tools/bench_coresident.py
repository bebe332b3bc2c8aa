"""Experiment (GPU box only): can the whitening pass K3 run UNDER the bilateral kernel K2, on the registers and shared
memory K2's two 288-thread blocks leave free on an SM (10240 registers)?  K3 is given a small-footprint geometry through
the tuning hook (generic row kernel, one vector per thread: 56 registers x (nt + 32) threads) and the bilateral WOW call
is timed with the side-stream overlap on.

    python tools/bench_coresident.py [--reps 20]"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import wavelets_b200 as wb  # noqa: E402
from wavelets_b200 import _lib  # noqa: E402
from tools.bench_wow import solar_like_device, timed  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--side", type=int, default=4096)
    args = ap.parse_args()
    lib = _lib.load(require_cuda=True)
    solar = solar_like_device(args.side, torch.float32)
    out = {}

    def run(tag):
        out[tag + "_bil_den_ms"] = timed(lambda: wb.wow(solar, bilateral=1, denoise_coefficients=[5, 2]), args.reps)
        out[tag + "_bil_ms"] = timed(lambda: wb.wow(solar, bilateral=1), args.reps)
        print(tag, {k: round(v, 4) for k, v in out.items() if k.startswith(tag)}, flush=True)

    for s in range(10):
        lib.wb_tune_k1(s, 0, 0, 0, 0)
    run("k3lean")
    for nt, ng, slots in ((128, 1, 6), (96, 1, 6), (64, 1, 6), (128, 1, 8), (256, 1, 6)):
        for s in range(10):
            lib.wb_tune_k1(s, nt, ng, slots, 0)
        run(f"k3nt{nt}ng{ng}s{slots}")
    for s in range(10):
        lib.wb_tune_k1(s, 0, 0, 0, 0)
    os.makedirs("gpurun_out", exist_ok=True)
    with open("gpurun_out/r2_coresident.json", "w") as fh:
        json.dump(out, fh, indent=1)


if __name__ == "__main__":
    main()
