"""wow() with a per-pixel noise map: the map cascade against the unfused route it replaces (needs a CUDA device).

    python tools/bench_noise_map.py [--side 4096] [--reps 10] [--out FILE.json]

Frame: solar_like(side, flux=1) in float32, noise map sqrt(frame) + 1, denoise_coefficients=[5, 2], plain and
bilateral=1.  Timed with CUDA events after a warm-up, the two sides alternating call by call:
  * "unfused": the route wow(noise=map) took before the map mode of the whitening kernel, rebuilt from public entry
    points -- the transform, then per thresholded scale K3 (sig_mode 0) into a temporary, Coefficients.significance
    with the map and the float64 product, per other scale K3 and a copy; the residual rescale and the synthesis;
  * "map": wow(img, noise=map) (one wb_wow_cascade_map call);
  * wow_batch of 8 frames with one map per frame against 8 wow() calls;
  * per thresholded scale, one K3 launch in map mode against one K3 launch with a scalar noise (soft).
Every pair of outputs is checked bit for bit.  Prints the GPU name and power limit; writes JSON only with --out."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import wavelets_b200 as wb  # noqa: E402
from oracle import atrous_oracle as orc  # noqa: E402
from wavelets_b200 import _lib, utils  # noqa: E402
from wavelets_b200.wavelets import _Noise, plane_moments, synthesis  # noqa: E402

DNS = [5, 2]


def unfused_map_route(img, nmap, bilateral):
    """wow(img, noise=nmap, denoise_coefficients=DNS, bilateral=...) the way the parent commit computed it."""
    lib = _lib.load(require_cuda=True)
    n_scales, sigma_bilateral, wts, dns = utils._wow_plan(img.shape, wb.B3spline, None, [], DNS, bilateral)
    co = wb.AtrousTransform(wb.B3spline, bilateral=sigma_bilateral)(img, n_scales)
    co.noise = nmap
    data, sf = co.data, co.scaling_function
    tmp = torch.empty_like(data[0])
    for s in range(n_scales):
        plane = data[s]
        utils._whiten_scale(lib, plane, tmp, s, sf, 0, 0.0, 1.0, _Noise(), wts[s])
        if dns[s] != 0:
            sig = co.significance(dns[s], s)
            plane.copy_((tmp.to(torch.float64) * sig.to(torch.float64)).to(plane.dtype))
        else:
            plane.copy_(tmp)
    last = data[n_scales]
    mom = plane_moments(last)
    _lib.check(lib.wb_residual_rescale(last.data_ptr(), last.numel(), 1, 0, _lib.dtype_code(last.dtype),
                                       mom.data_ptr(), float(wts[n_scales]), _lib.stream_ptr(last.device)))
    return synthesis(data), data


def alternate(fns, reps, warmup=2):
    """Milliseconds per call of each function (median over reps), calls alternating, CUDA events around each."""
    for _ in range(warmup):
        for f in fns:
            f()
    times = [[] for _ in fns]
    for _ in range(reps):
        for i, f in enumerate(fns):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            f()
            b.record()
            b.synchronize()
            times[i].append(a.elapsed_time(b))
    return [float(np.median(t)) for t in times]


def same_bits(a, b):
    v = torch.int32 if a.dtype == torch.float32 else torch.int64
    return a.shape == b.shape and bool(torch.equal(a.view(v), b.view(v)))


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--side", type=int, default=4096)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--out", default=None, help="also write the results as JSON to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_noise_map.py needs a CUDA device")
    res = {**gpu_info(), "side": args.side, "dtype": "float32", "denoise_coefficients": DNS, "ms": {},
           "bit_identical": {}}
    print(res["device"], "|", res["nvidia_smi"], flush=True)
    frame = orc.solar_like(args.side, seed=2, flux=1, dtype=np.float32)
    img = torch.from_numpy(frame).cuda()
    nmap = torch.from_numpy(np.sqrt(frame) + 1).cuda()
    lib = _lib.load(require_cuda=True)
    for bil in (None, 1):
        tag = "plain" if bil is None else "bilateral"
        r0, p0 = unfused_map_route(img, nmap, bil)
        r1, co = wb.wow(img, noise=nmap, denoise_coefficients=DNS, bilateral=bil)
        ok = same_bits(r0, r1) and same_bits(p0, co.data)
        res["bit_identical"][f"wow_{tag}"] = ok
        t_old, t_new = alternate([lambda: unfused_map_route(img, nmap, bil),
                                  lambda: wb.wow(img, noise=nmap, denoise_coefficients=DNS, bilateral=bil)], args.reps)
        res["ms"][f"wow_{tag}"] = {"unfused": t_old, "map": t_new}
        print(f"wow {tag:9s}: unfused {t_old:8.3f} ms   map {t_new:8.3f} ms   bit-identical {ok}", flush=True)
        # a stack of frames with one map each against one wow() per frame
        side_b = args.side // 2
        frames = torch.stack([torch.from_numpy(orc.solar_like(side_b, seed=10 + i, flux=1, dtype=np.float32))
                              for i in range(args.batch)]).cuda()
        maps = torch.sqrt(frames) + 1
        rb, pb, _ = wb.wow_batch(frames, noise=maps, denoise_coefficients=DNS, bilateral=bil)
        ok = all(same_bits(rb[i], wb.wow(frames[i], noise=maps[i], denoise_coefficients=DNS, bilateral=bil)[0])
                 for i in range(args.batch))
        res["bit_identical"][f"batch_{tag}"] = ok

        def singles():
            for i in range(args.batch):
                wb.wow(frames[i], noise=maps[i], denoise_coefficients=DNS, bilateral=bil)
        t_b, t_s = alternate([lambda: wb.wow_batch(frames, noise=maps, denoise_coefficients=DNS, bilateral=bil),
                              singles], args.reps)
        res["ms"][f"batch{args.batch}_{side_b}_{tag}"] = {"wow_batch": t_b, "wow_per_frame": t_s}
        print(f"{args.batch} x {side_b}^2 {tag:9s}: wow_batch {t_b:8.3f} ms   {args.batch} wow() {t_s:8.3f} ms   "
              f"bit-identical {ok}", flush=True)
    # one K3 launch per thresholded scale: map mode against a scalar noise (soft threshold)
    sf = wb.B3spline(2)
    h = w = args.side
    code = _lib.dtype_code(img.dtype)
    st = _lib.stream_ptr(img.device)
    _, raw = wb.atrous_scale(img, 0, sf)
    out = torch.empty_like(raw)
    sigma_e = sf.sigma_e()
    for s in range(len(DNS)):
        _, raw = wb.atrous_scale(img, s, sf)

        def k3_map():
            _lib.check(lib.wb_wow_whiten_scale_map(raw.data_ptr(), out.data_ptr(), nmap.data_ptr(), 1, h, w, w, 0, w, 0,
                                                   w, 0, s, sf.taps_code, code, 1, float(DNS[s]), float(sigma_e[s]),
                                                   1.0, st))

        def k3_scalar():
            _lib.check(lib.wb_wow_whiten_scale(raw.data_ptr(), out.data_ptr(), 1, h, w, w, 0, w, 0, s, sf.taps_code, code,
                                               1, float(DNS[s]), float(sigma_e[s]), 40.0, None, 1.0, st))
        t_m, t_s = alternate([k3_map, k3_scalar], 5 * args.reps)
        bytes_map, bytes_scalar = 3 * 4 * h * w, 2 * 4 * h * w
        res["ms"][f"k3_scale{s}"] = {"map": t_m, "scalar_soft": t_s,
                                     "map_TB_per_s": bytes_map / t_m / 1e9, "scalar_TB_per_s": bytes_scalar / t_s / 1e9}
        print(f"K3 scale {s}: map {1e3 * t_m:7.1f} us ({bytes_map / t_m / 1e9:.2f} TB/s of 12 B/px)   "
              f"scalar soft {1e3 * t_s:7.1f} us ({bytes_scalar / t_s / 1e9:.2f} TB/s of 8 B/px)", flush=True)
    assert all(res["bit_identical"].values()), res["bit_identical"]
    if args.out is not None:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
