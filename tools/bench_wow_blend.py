"""wow() with the gamma blend and preserve_variance: one wb_wow_cascade_blend call against the element-wise route it
replaces (needs a CUDA device).

    python tools/bench_wow_blend.py [--reps 10] [--out FILE.json]

Options h=0.9, denoise_coefficients=[5, 2] on solar_like(side, flux=1) frames.  Timed with CUDA events after a warm-up,
the two sides alternating call by call:
  * "parent": the route wow() took before, rebuilt from the code that stays in the tree -- AtrousTransform, then
    _wow_general plane by plane (K3, wb_denoise_plane, torch element-wise ops for the gamma plane and the blend);
  * "blend": wow() (one wb_wow_cascade_blend call);
at 1024^2, 2048^2, 4096^2 float32, 4096^2 bilateral, 4096^2 float64; wow_batch of 16 x 2048^2 against 16 parent calls;
wow_stream of 16 host frames of 4096^2 against the bare host -> device -> host copy of the same frames, upload
and download overlapped (the ceiling),
and against the parent route frame by frame.  Every pair of outputs is checked bit for bit.

Byte model (HBM traffic in units of T = sizeof(dtype) per pixel, L scales, k thresholded scales; the MAD estimate is
left out, both routes pay it):
  * blend:  per scale K1 3 (read c_s, write c_s+1 and w_s) + K3 2 + epilogue 3 (read w_s and gamma, write gamma;
    2 at scale 0), moments of c_L 1, residual 4, synthesis + blend L + 3  ->  9 L + 7   (97 at L = 10)
  * parent: transform 3 L, per scale K3 2 + gamma += 3 + copy 2 (+ 2 for wb_denoise_plane where thresholded), residual
    moments 1 + gamma += 3 + mul_ 2, synthesis L + 2, min + max 2, -= /= clamp_ pow_ 8, the blend 7
    ->  11 L + 2 k + 25   (139 at L = 10, k = 2)
Prints the GPU name and power limit; writes JSON only with --out."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import wavelets_b200 as wb  # noqa: E402
from oracle import atrous_oracle as orc  # noqa: E402
from wavelets_b200 import utils  # noqa: E402

KW = dict(h=0.9, denoise_coefficients=[5, 2])


def parent_route(img, **kw):
    """wow(img, **kw) for a 2-D image with h != 0 or preserve_variance, as the parent commit computed it."""
    kw = dict(KW, **kw)
    n_scales, sigma_bilateral, wts, dns = utils._wow_plan(img.shape, wb.B3spline, None, [], kw["denoise_coefficients"],
                                                          kw.get("bilateral"), h=kw["h"])
    co = wb.AtrousTransform(wb.B3spline, bilateral=sigma_bilateral)(img, n_scales)
    co.noise = None
    return utils._wow_general(co, [], True, kw["denoise_coefficients"], kw.get("bilateral"), True, False, 3.2, None,
                              None, kw["h"], plan=(n_scales, wts, dns))


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


def byte_model(L, k):
    return {"blend": 9 * L + 7, "parent": 11 * L + 2 * k + 25}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None, help="also write the results as JSON to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_wow_blend.py needs a CUDA device")
    res = {**gpu_info(), "options": KW, "ms": {}, "bit_identical": {}, "hbm_fraction": {}}
    print(res["device"], "|", res["nvidia_smi"], flush=True)
    peak = 7.7e12  # B/s, HBM3e of one B200 (data sheet): the fraction below is bytes of the model / time / this
    for tag, side, dt, extra in (("1024", 1024, np.float32, {}), ("2048", 2048, np.float32, {}),
                                 ("4096", 4096, np.float32, {}), ("4096_bilateral", 4096, np.float32, {"bilateral": 1}),
                                 ("4096_f64", 4096, np.float64, {})):
        img = torch.from_numpy(orc.solar_like(side, seed=2, flux=1, dtype=dt)).cuda()
        r0, c0 = parent_route(img, **extra)
        r1, c1 = wb.wow(img, **KW, **extra)
        ok = same_bits(r0, r1) and same_bits(c0.data, c1.data)
        res["bit_identical"][tag] = ok
        t_old, t_new = alternate([lambda: parent_route(img, **extra), lambda: wb.wow(img, **KW, **extra)], args.reps)
        L = len(c1) - 1
        model = byte_model(L, sum(1 for d in KW["denoise_coefficients"][:L] if d))
        es = img.element_size() * side * side
        frac = {k: model[k] * es / (t * 1e-3) / peak for k, t in (("parent", t_old), ("blend", t_new))}
        res["ms"][tag] = {"parent": t_old, "blend": t_new, "speedup": t_old / t_new, "L": L, "bytes_model_T": model}
        res["hbm_fraction"][tag] = frac
        print(f"wow {tag:15s}: parent {t_old:8.3f} ms ({model['parent']} T, {frac['parent']:.2f} of HBM)   "
              f"blend {t_new:8.3f} ms ({model['blend']} T, {frac['blend']:.2f})   x{t_old / t_new:.2f}   "
              f"bit-identical {ok}", flush=True)
    # a stack: one wow_batch call against one parent route per frame
    n_b, side_b = 16, 2048
    frames = torch.stack([torch.from_numpy(orc.solar_like(side_b, seed=10 + i, flux=1, dtype=np.float32))
                          for i in range(n_b)]).cuda()
    rb, _, _ = wb.wow_batch(frames, **KW)
    ok = all(same_bits(rb[i], parent_route(frames[i])[0]) for i in range(n_b))
    res["bit_identical"]["batch"] = ok

    def parent_frames():
        for i in range(n_b):
            parent_route(frames[i])
    t_p, t_b = alternate([parent_frames, lambda: wb.wow_batch(frames, **KW)], max(3, args.reps // 2), warmup=1)
    res["ms"][f"batch{n_b}_{side_b}"] = {"parent_per_frame": t_p / n_b, "wow_batch_per_frame": t_b / n_b}
    print(f"{n_b} x {side_b}^2: parent {t_p / n_b:8.3f} ms/frame   wow_batch {t_b / n_b:8.3f} ms/frame   "
          f"bit-identical {ok}", flush=True)
    del frames, rb
    # host frames: wow_stream against the bare copy ceiling and the parent route frame by frame
    n_s, side_s = 16, 4096
    host = torch.stack([torch.from_numpy(orc.solar_like(side_s, seed=20 + i, flux=1, dtype=np.float32))
                        for i in range(4)]).repeat(n_s // 4, 1, 1).pin_memory()
    out = torch.empty_like(host).pin_memory()
    d_buf = torch.empty((side_s, side_s), dtype=torch.float32, device="cuda")
    d_two = [torch.empty_like(d_buf) for _ in range(2)]
    s_up, s_down = torch.cuda.Stream(), torch.cuda.Stream()
    ev_up = [torch.cuda.Event() for _ in range(2)]
    ev_down = [torch.cuda.Event() for _ in range(2)]

    def bare_copy():
        """The upload of frame i+1 under the download of frame i, two device buffers: what a stream can reach."""
        for i in range(n_s):
            k = i % 2
            with torch.cuda.stream(s_up):
                if i >= 2:
                    s_up.wait_event(ev_down[k])
                d_two[k].copy_(host[i], non_blocking=True)
                ev_up[k].record(s_up)
            with torch.cuda.stream(s_down):
                s_down.wait_event(ev_up[k])
                out[i].copy_(d_two[k], non_blocking=True)
                ev_down[k].record(s_down)
        torch.cuda.synchronize()

    def parent_stream():
        for i in range(n_s):
            d_buf.copy_(host[i], non_blocking=True)
            out[i].copy_(parent_route(d_buf)[0], non_blocking=True)
        torch.cuda.synchronize()

    def stream():
        wb.wow_stream(host, out=out, **KW)
    stream()
    ok = all(same_bits(out[i].cuda(), parent_route(host[i].cuda())[0]) for i in range(4))
    res["bit_identical"]["stream"] = ok
    t = {}
    for name, f in (("bare_copy", bare_copy), ("parent_per_frame", parent_stream), ("wow_stream", stream)):
        f()
        samples = []
        for _ in range(3):
            t0 = time.perf_counter()
            f()
            samples.append((time.perf_counter() - t0) * 1e3 / n_s)
        t[name] = float(np.median(samples))
    res["ms"][f"stream{n_s}_{side_s}"] = t
    print(f"stream {n_s} x {side_s}^2 host frames: bare copy {t['bare_copy']:7.3f} ms/frame   parent "
          f"{t['parent_per_frame']:7.3f}   wow_stream {t['wow_stream']:7.3f}   bit-identical {ok}", flush=True)
    assert all(res["bit_identical"].values()), res["bit_identical"]
    if args.out is not None:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
