"""Volumes (D, H, W): the per-scale route (wb_atrous_scale + wb_atrous_axis, and _wow_nd's element-wise loop) against
wb_atrous_transform_volume / wb_wow_cascade_volume, alternated in one process and timed with CUDA events.

    python -m tools.bench_volume [--reps 5] [--out profiles/r4_bench_volume.json]

Cubes: fp32 128 x 2048^2 and 64 x 4096^2, fp64 128 x 2048^2 (2 - 4 GiB per volume, far beyond the 126 MB L2, so every
pass streams from HBM).  Algorithmic bytes per call, in volumes of D*H*W elements: the transform reads c_s and writes
c_{s+1} and w_s (3 per scale); wow() adds the whitening of every plane (read + write, 2 per scale), the residual
rescale (moments read + rescale read/write: 3) and the synthesis (L + 1 reads, 1 write).  Peak memory is
torch.cuda.max_memory_allocated above what was allocated before the call."""
import argparse
import json
import subprocess
import sys

import torch

import wavelets_b200 as wb
from wavelets_b200 import utils, wavelets


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[torch.cuda.current_device()] if q.returncode == 0 else "unknown"


def timed(fn, reps):
    """Median device time (ms) of fn over reps calls, and the peak memory above the starting allocation (bytes)."""
    times = []
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
        del out
    peak = torch.cuda.max_memory_allocated() - base
    times.sort()
    return times[len(times) // 2], peak


def old_transform(vol, level):
    return wb.AtrousTransform(wb.B3spline)._run_nd_reference(vol, level, wb.B3spline(3))


def new_transform(vol, level):
    return wb.AtrousTransform(wb.B3spline)(vol, level).data


def old_wow(vol, dns):
    return utils_ref_wow(vol, dns)


def utils_ref_wow(vol, dns):
    L, _, wts, dn = utils._wow_plan(vol.shape, wb.B3spline, None, [], dns, None, n_dims=3)
    co = wavelets.Coefficients(old_transform(vol, L), wb.B3spline(3), None)
    return utils._wow_nd(co, wts, dn, True, True, False, 3.2, None, None, 0, smooth=wavelets._smooth_nd_reference), co


def new_wow(vol, dns):
    return wb.wow(vol, denoise_coefficients=dns)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    ap.add_argument("--small", action="store_true", help="tiny cubes (a dry run of the script)")
    args = ap.parse_args()
    torch.cuda.set_device(0)
    cases = [("fp32", torch.float32, (128, 2048, 2048)), ("fp32", torch.float32, (64, 4096, 4096)),
             ("fp64", torch.float64, (128, 2048, 2048))]
    if args.small:
        cases = [("fp32", torch.float32, (16, 64, 64))]
    dns = [3, 1]
    result = {"card": card(), "reps": args.reps, "timer": "CUDA events, median", "cases": []}
    for name, dt, shape in cases:
        vol = torch.randn(shape, dtype=dt, device="cuda") * 0.5 + 2.0
        es = vol.element_size()
        nv = vol.numel() * es
        L = utils._wow_plan(shape, wb.B3spline, None, [], dns, None, n_dims=3)[0]
        # bit-identity of the two routes on this cube, once
        assert torch.equal(old_transform(vol, L), new_transform(vol, L))
        r_old, co_old = old_wow(vol, dns)
        r_new, co_new = new_wow(vol, dns)
        assert torch.equal(r_old, r_new) and torch.equal(co_old.data, co_new.data)
        del r_old, co_old, r_new, co_new
        bytes_t = 3 * L * nv
        bytes_w = (3 * L + 2 * L + 3 + L + 2) * nv
        rows = {}
        for op, fns, nbytes in (("transform", (lambda: old_transform(vol, L), lambda: new_transform(vol, L)), bytes_t),
                                ("wow", (lambda: old_wow(vol, dns), lambda: new_wow(vol, dns)), bytes_w)):
            acc = {"old": [], "new": []}
            peaks = {}
            for _ in range(2):  # alternate the two routes
                for tag, fn in zip(("old", "new"), fns):
                    fn()  # warm-up of this shape
                    t, pk = timed(fn, args.reps)
                    acc[tag].append(t)
                    peaks[tag] = max(peaks.get(tag, 0), pk)
            row = {"algorithmic_bytes": nbytes}
            for tag in ("old", "new"):
                t = min(acc[tag])
                row[tag] = {"ms": round(t, 3), "GB_per_s": round(nbytes / t / 1e6, 1), "peak_bytes": peaks[tag]}
            row["speedup"] = round(row["old"]["ms"] / row["new"]["ms"], 2)
            rows[op] = row
        case = {"dtype": name, "shape": list(shape), "n_scales": L, "denoise_coefficients": dns, **rows}
        result["cases"].append(case)
        print(json.dumps(case), flush=True)
        del vol
        torch.cuda.empty_cache()
    print(json.dumps({"card": result["card"]}))
    if args.out:
        with open(args.out, "w") as fh:
            json.dump(result, fh, indent=1)
    return 0


if __name__ == "__main__":
    sys.exit(main())
