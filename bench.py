#!/usr/bin/env python
"""Benchmark of the à trous hot path on B200 (see DESIGN.md section "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--no-wow] [--no-extras]
                    [--dump-outputs DIR]

Workload at N=1 (BASELINE.json configs[1]): B3spline 2-D à trous transform of one 4096x4096 fp32 frame over 10
scales.  One "step" = one full transform (10 per-scale launches) of a device-resident frame; `value` is
Mpixel*scales/s over all ranks (weak scaling: every rank transforms its own frame).  `e2e` is the same metric
through the public Python API with HOST buffers (AtrousTransform.stream): pinned-host -> device copy of the frame,
transform, device -> pinned-host copy of all 11 planes, every step, consecutive steps overlapped on three streams.  `roofline` is for the dominant kernel (atrous_rows_kernel):
algorithmic bytes 3*sizeof(T) per pixel per launch / measured launch time, against MEASURED_PEAKS.json.
`cpu_baseline` / `--impl reference` time the reference's own CPU algorithm (oracle port: the same cv2.filter2D
calls the reference makes) on the host cores.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_SIDE = 4096
LEVELS = 10
SF_NAME = "b3spline"
METRIC = "atrous_transform_throughput"
UNIT = "Mpixel*scales/s"
WORKLOAD = "cfg2: B3spline 2-D a trous, 4096x4096 fp32, 10 scales (BASELINE.json configs[1])"
# The SAME dict in both arms' lines (the driver compares them key by key); per-arm details go to "detail".
CONFIG = {"workload": WORKLOAD, "scaling_function": "b3spline", "side": N_SIDE, "scales": LEVELS, "frames_per_rank": 1,
          "sharding": "one frame per rank, no collective",
          "l2": "working set 14 planes x 64 MiB = 896 MiB per step >> 126 MB L2 (no flush needed)"}


def measured_peaks():
    """HBM roofline denominator: the driver-written MEASURED_PEAKS.json (the SUSTAINED figure when the file tells burst
    and sustained apart -- K1 is timed inside a long step), else the fallback of B200_PROFILING.md."""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            with open(path) as fh:
                d = json.load(fh)

            def num(v):
                if isinstance(v, (int, float)) and v > 0:
                    return float(v)
                if isinstance(v, dict):
                    for k in ("sustained", "sustained_gbs", "gbs", "value", "burst"):
                        if k in v and isinstance(v[k], (int, float)) and v[k] > 0:
                            return float(v[k])
                return None

            for key in ("hbm_gbs_sustained", "hbm_sustained_gbs", "hbm_gbs"):
                if key in d and num(d[key]):
                    return num(d[key]), f"MEASURED_PEAKS.json[{key}] (of measured)"
            for key, v in d.items():
                if "hbm" in key.lower() and "burst" not in key.lower() and num(v):
                    return num(v), f"MEASURED_PEAKS.json[{key}] (of measured)"
        except (OSError, ValueError):
            pass
    return 6650.0, "B200_PROFILING.md fallback (of fallback)"


def ncu_traffic():
    """Per-launch DRAM bytes of the dominant kernel from the committed ncu capture (profiles/), or None."""
    path = os.path.join(ROOT, "profiles", "k1_traffic.json")
    if os.path.exists(path):
        with open(path) as fh:
            return json.load(fh).get("dram_bytes_per_launch")
    return None


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons through NVML while the timed region runs."""

    def __init__(self, index, uuid=None, period=0.02):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop_evt = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            try:  # robust against CUDA_VISIBLE_DEVICES renumbering
                self.h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + str(uuid)).encode())
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def cpu_reference_rate(side, levels, repeats=1):
    """Mpixel*scales/s of the reference's CPU algorithm (oracle port; cv2 backend = the reference's own calls)."""
    from oracle import atrous_oracle as orc
    backend = orc.default_backend()
    img = np.random.default_rng(0).standard_normal((side, side)).astype(np.float32)
    best = None
    for _ in range(repeats):
        t0 = time.perf_counter()
        orc.atrous_transform(img, levels, SF_NAME, backend=backend)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    threads = 1
    if backend == "cv2":
        import cv2
        threads = cv2.getNumThreads()
    return side * side * levels / best / 1e6, best, backend, threads


DUMP_SAMPLES = 1 << 20  # pixel positions kept per plane: 11 planes x 2^20 x 4 B = 44 MiB


def dump_outputs(out_dir, planes):
    """Writes out_dir/planes_sample.npy: the (LEVELS + 1) planes of one transform at a fixed, seeded sample of
    DUMP_SAMPLES pixel positions (the same positions in every plane, in row-major order), as a float32 or float64
    (LEVELS + 1, DUMP_SAMPLES) array.  The positions depend only on the frame size, so two builds run with the same
    arguments can be compared value for value."""
    n = planes.shape[-2] * planes.shape[-1]
    idx = np.sort(np.random.default_rng(0).choice(n, size=min(DUMP_SAMPLES, n), replace=False))
    flat = planes.reshape(planes.shape[0], n)
    if isinstance(flat, np.ndarray):
        sample = flat[:, idx]
    else:  # torch tensor on the device: gather there, copy only the sample
        import torch
        sample = flat[:, torch.from_numpy(idx).to(flat.device)].cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "planes_sample.npy"), sample)


def run_reference(args):
    """--impl reference: the reference's CPU path (oracle port) on the host cores; rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import atrous_oracle as orc
    backend = orc.default_backend()
    # Bounded sample: FULL-SIZE frames of the named workload, as many of the K requested steps as fit in ~100 s of CPU
    # work.  A crop would not be a sample of the same workload: the reference convolves with the dense dilated kernel
    # (2049 x 2049 taps at scale 9) through a DFT whose cost hardly depends on the image size (measured here: 1.7 / 4.5
    # / 8.4 Mpixel*scales/s on 256^2 / 512^2 / 1024^2 crops against 29 on the 4096^2 frame), so shrinking the frame to
    # fit K steps would understate the reference by an order of magnitude.
    side = N_SIDE
    img = np.random.default_rng(0).standard_normal((side, side)).astype(np.float32)
    t0 = time.perf_counter()
    orc.atrous_transform(img, LEVELS, SF_NAME, backend=backend)  # first warm-up frame (~6 s each)
    t_frame = time.perf_counter() - t0
    # W warm-up frames and K timed steps are honoured exactly while they fit in ~5 minutes of CPU work (W + K <= ~50 at
    # 5.7 s per frame: the driver's W = 5, K = 20 take ~2.5 minutes); beyond that the warm-up stops at half a minute and
    # every step is accounted at the mean time of a bounded sample of full frames (both stated in `sample`).
    warm = max(1, min(int(args.warmup), int(60.0 / max(t_frame, 1e-3)))) if (args.warmup + args.steps) * t_frame > 300.0 \
        else max(1, int(args.warmup))
    for _ in range(warm - 1):
        orc.atrous_transform(img, LEVELS, SF_NAME, backend=backend)
    timed = max(1, min(args.steps, int(240.0 / max(t_frame, 1e-3))))
    t0 = time.perf_counter()
    for _ in range(timed):
        planes = orc.atrous_transform(img, LEVELS, SF_NAME, backend=backend)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, planes)
    value = side * side * LEVELS * timed / dt / 1e6
    threads = 1
    if backend == "cv2":
        import cv2
        threads = cv2.getNumThreads()
    sample = (f"{timed} full {side}x{side} fp32 frames x {LEVELS} scales timed"
              + ("" if timed == args.steps else f" (bounded sample: {args.steps} steps requested, each accounted at the mean)")
              + f", {warm} warm-up frame(s), oracle port backend={backend} = the reference's own cv2.filter2D calls")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "steps_timed": timed, "warmup": args.warmup, "warmup_done": warm, "ms_per_step": dt / timed * 1e3,
        "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": dict(CONFIG),
        "detail": {"sample": sample},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def solar_like_device(n, dtype, device, seed=2, flux=0.05):
    """Synthetic solar-like frame generated on the device (SURVEY.md 8(d) 'S': limb-darkened disk + exponential corona
    + 30 Gaussian active regions + background, photon noise, integer counts)."""
    import torch
    g = torch.Generator(device=device).manual_seed(seed)
    ax = torch.arange(n, device=device, dtype=torch.float64)
    y, x = torch.meshgrid(ax, ax, indexing="ij")
    r = torch.hypot(x - n / 2, y - n / 2) / (0.4 * n)
    img = torch.where(r < 1, 2000 * (0.4 + 0.6 * torch.sqrt(torch.clamp(1 - r ** 2, min=0))),
                      800 * torch.exp(-(torch.clamp(r, min=1) - 1) / 0.15))
    for _ in range(30):
        cx, cy = ((torch.rand(2, generator=g, device=device) * 0.6 + 0.2) * n).tolist()
        sg = float(torch.rand(1, generator=g, device=device) * 27 + 3) * n / 1024
        amp = float(torch.rand(1, generator=g, device=device) * 7500 + 500)
        img += amp * torch.exp(-((x - cx) ** 2 + (y - cy) ** 2) / (2 * sg ** 2))
    img = (img + 20) * flux
    img = img + torch.sqrt(img) * torch.randn(img.shape, generator=g, device=device, dtype=torch.float64)
    return torch.round(torch.clamp(img, min=0)).to(dtype)


def time_wow(wb, img, reps, peak, **kw):
    """Device-resident wow(): frames/s and the algorithmic-byte roofline of SURVEY.md 8(d), (5L+3)*sizeof(T) B/pixel."""
    import torch
    for _ in range(3):
        _, co = wb.wow(img, **kw)
    levels = len(co) - 1
    del co
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        wb.wow(img, **kw)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    algo = (5 * levels + 3) * img.element_size() * img.numel()
    return {"frames_per_s": 1e3 / ms, "ms_per_frame": ms, "scales": levels, "algorithmic_bytes_per_frame": algo,
            "achieved_gbs": algo / ms / 1e6, "frac_of_hbm_peak": algo / ms / 1e6 / peak}


def pin_to_gpu_numa_node(index, uuid=None):
    """Bind this process to the CPUs NVML reports as local to the GPU BEFORE any pinned allocation: first-touch then
    places the pinned buffers on the GPU's own NUMA node (8 ranks otherwise share one node's memory controller and
    PCIe root for their host copies).  Returns the number of CPUs bound, or None when NVML cannot tell."""
    try:
        import pynvml
        pynvml.nvmlInit()
        try:
            h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + str(uuid)).encode())
        except Exception:
            h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * i + b for i, wd in enumerate(mask) for b in range(64) if (wd >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


def copy_ceiling(dev, h2d_bytes, d2h_bytes, barrier, reps=4):
    """What plain pinned copies of one step's bytes reach on this box with every rank copying at once (H2D and D2H on
    two streams, device time): the ceiling of the e2e number at this N."""
    import torch
    hin = torch.empty(h2d_bytes, dtype=torch.uint8).pin_memory()
    hout = torch.empty(d2h_bytes, dtype=torch.uint8).pin_memory()
    din = torch.empty(h2d_bytes, dtype=torch.uint8, device=dev)
    dout = torch.empty(d2h_bytes, dtype=torch.uint8, device=dev)
    s1, s2 = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    cur = torch.cuda.current_stream(dev)

    def once():
        s1.wait_stream(cur)
        s2.wait_stream(cur)
        with torch.cuda.stream(s1):
            din.copy_(hin, non_blocking=True)
        with torch.cuda.stream(s2):
            hout.copy_(dout, non_blocking=True)
        cur.wait_stream(s1)
        cur.wait_stream(s2)

    once()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(cur)
    for _ in range(reps):
        once()
    e1.record(cur)
    barrier()
    return e0.elapsed_time(e1) / reps


def multi_gpu_extras(args, wb, dist, dev, rank, world, peak):
    """The modes with more than one frame per job (N > 1 only): cfg4 (frames sharded, no collective) and cfg5 (ONE image
    in N row bands, per-scale halo transfer over NVLink).  Every number: device events, max over ranks."""
    import torch
    from wavelets_b200.sharded import BandedTransform, band_range, halo_rows
    out = {}

    def barrier():
        dist.barrier()
        torch.cuda.synchronize(dev)

    def max_ms(ms):
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    # ---- cfg4: batch of 4096^2 frames, B3spline 8 scales + WOW, frames dealt to the ranks (weak scaling) -------------
    nb, L4, reps4 = 16, 8, 4
    frame = solar_like_device(N_SIDE, torch.float32, dev, seed=3 + rank)
    stack = frame.unsqueeze(0).repeat(nb, 1, 1)
    stack += torch.sqrt(stack.clamp(min=1)) * 0.1 * torch.randn(stack.shape, device=dev)
    for _ in range(2):
        wb.wow_batch(stack, n_scales=L4)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps4):
        wb.wow_batch(stack, n_scales=L4)
    e1.record()
    barrier()
    ms = max_ms(e0.elapsed_time(e1))
    algo4 = (5 * L4 + 3) * 4 * N_SIDE * N_SIDE
    fps = world * nb * reps4 / (ms / 1e3)
    out["wow_batch_cfg4"] = {
        "frames_per_s": fps, "frames_per_s_per_gpu": fps / world, "ms_per_frame_per_gpu": ms / (nb * reps4), "scales": L4,
        "frames_per_rank": nb * reps4, "frames_per_launch": nb, "sharding": "frames dealt to the ranks, no collective",
        "algorithmic_bytes_per_frame": algo4, "frac_of_hbm_peak": algo4 * fps / world / 1e9 / peak,
        "call": f"wow_batch({nb} x 4096x4096 fp32 solar-like, n_scales=8) per rank, BASELINE.json configs[3]"}
    del stack, frame
    torch.cuda.empty_cache()

    # ---- cfg5: ONE 32768^2 image, B3spline 12 scales, N row bands ------------------------------------------------------
    def run_banded(side, levels, reps, check):
        y0, y1 = band_range(side, rank, world)
        res = {}
        gen = torch.Generator(device=dev).manual_seed(99)
        full = None
        if check:
            img = torch.randn((side, side), generator=gen, device=dev, dtype=torch.float32)
            band = img[y0:y1].contiguous()
            full = wb.AtrousTransform(wb.B3spline)(img, levels).data[:, y0:y1].clone()
            del img
        else:
            gen.manual_seed(99 + rank)
            band = torch.randn((y1 - y0, side), generator=gen, device=dev, dtype=torch.float32)
        for mode in ("push", "nccl"):
            bt = BandedTransform(wb.B3spline, push=(mode == "push"))
            planes = bt(band, levels, side)
            if full is not None:
                flag = torch.tensor([1 if torch.equal(planes, full) else 0], device=dev)
                dist.all_reduce(flag, op=dist.ReduceOp.MIN)
                res[f"bit_identical_{mode}"] = bool(flag.item())
            del planes
            bt(band, levels, side)
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                bt(band, levels, side)
            e1.record()
            barrier()
            ms = max_ms(e0.elapsed_time(e1) / reps)
            res[mode] = {"ms": ms, "mpx_scales_per_s": side * side * levels / ms / 1e3}
        del band, full
        torch.cuda.empty_cache()
        return res

    side5, L5 = 32768, 12
    chk = run_banded(16384, 11, 3, True)      # fits one GPU: every rank also runs the unsharded cascade and compares
    big = run_banded(side5, L5, 3, False)
    rows = side5 // world
    halo_bytes = [2 * min(halo_rows(s, 5), rows) * side5 * 4 for s in range(L5)]  # ingress per interior rank per scale
    best = min(("push", "nccl"), key=lambda m: big[m]["ms"])
    hbm_ms = L5 * 3 * 4 * rows * side5 / (peak * 1e9) * 1e3
    link_ms = sum(halo_bytes) / 770e9 * 1e3
    out["banded"] = {
        "call": f"BandedTransform(B3spline)(band, 12, 32768): one 32768x32768 fp32 image in {world} row bands, "
                "BASELINE.json configs[4]",
        "ms": big[best]["ms"], "mpx_scales_per_s": big[best]["mpx_scales_per_s"], "transport": best,
        "ms_by_transport": {m: big[m]["ms"] for m in big},
        "transports": {"push": "halo rows of the next scale stored into the neighbours' buffers by the scale kernel "
                               "(posted NVLink writes from wb_atrous_scale_band_push), one device barrier per scale",
                       "nccl": "per-scale ncclSend/ncclRecv halo exchange, then the band kernel"},
        "halo_bytes_in_per_scale_interior_rank": halo_bytes, "halo_bytes_in_total": sum(halo_bytes),
        "floor_ms": {"hbm_3T_per_scale": hbm_ms, "nvlink_770GBs": link_ms,
                     "note": "transfers of scale s+1 cannot start before scale s is computed: the floor with in-kernel "
                             "overlap is the sum over scales of max(hbm, link), not max of the sums"},
        "bit_identical": bool(chk.get("bit_identical_push", False) and chk.get("bit_identical_nccl", False)),
        "bit_identical_check": {"image": "16384x16384 fp32, 11 scales, banded vs unsharded on every rank",
                                **{k: v for k, v in chk.items() if k.startswith("bit_identical")},
                                "ms": {m: chk[m]["ms"] for m in ("push", "nccl")}},
    }
    return out


def run_ours(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: wavelets_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    all_cpus = os.sched_getaffinity(0)
    numa_cpus = pin_to_gpu_numa_node(local_rank, getattr(torch.cuda.get_device_properties(dev), "uuid", None))

    import wavelets_b200 as wb
    from wavelets_b200 import _lib

    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load(require_cuda=True)

    h = w = N_SIDE
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    img = torch.randn((h, w), generator=gen, device=dev, dtype=torch.float32)
    planes = torch.empty((LEVELS + 1, h, w), dtype=torch.float32, device=dev)
    scratch = torch.empty((2, h, w), dtype=torch.float32, device=dev)
    stream = torch.cuda.current_stream(dev)
    assert lib.wb_atrous_scale_path(h, w, w, w, 0, _lib.WB_B3SPLINE, _lib.WB_F32, img.data_ptr(), scratch.data_ptr(),
                                    planes.data_ptr()) == 1, "expected the TMA row-pipeline kernel on this shape"

    def step():
        _lib.check(lib.wb_atrous_transform(img.data_ptr(), planes.data_ptr(), scratch.data_ptr(), 1, h, w, w, 0,
                                           LEVELS, _lib.WB_B3SPLINE, _lib.WB_F32, stream.cuda_stream))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    sampler = ClockSampler(local_rank, uuid=getattr(torch.cuda.get_device_properties(dev), "uuid", None))
    warmup = max(3, args.warmup)
    for _ in range(warmup):
        step()
    barrier()
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(stream)
    for _ in range(args.steps):
        step()
    e1.record(stream)
    barrier()
    elapsed_ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, planes)
    if args.steps * 0.4 < 300:  # short run: extend the sampling window with untimed identical steps
        t_end = time.perf_counter() + 0.5
        while time.perf_counter() < t_end:
            for _ in range(50):
                step()
            torch.cuda.synchronize(dev)
    clocks = sampler.stop()

    # ---- end-to-end through the public API with host buffers ------------------------------------------------
    e2e_steps = max(1, min(args.steps, 20))
    host_in = torch.randn((h, w), dtype=torch.float32).pin_memory()
    host_out = torch.empty((LEVELS + 1, h, w), dtype=torch.float32).pin_memory()
    transform = wb.AtrousTransform(wb.B3spline)

    # One step = one frame through AtrousTransform.stream(): pinned-host -> device copy of the frame, the transform,
    # device -> pinned-host copy of all 11 planes; consecutive steps overlap on three CUDA streams (the upload of step
    # n+1 and the kernels of step n hide behind the download of step n-1).  Every step re-reads the same host frame and
    # rewrites the same host planes (stride-0 views), so the pinned footprint stays at one frame + one set of planes.
    frames_view = host_in.unsqueeze(0).expand(e2e_steps, h, w)
    out_view = host_out.unsqueeze(0).expand(e2e_steps, LEVELS + 1, h, w)

    def e2e_run(n):
        transform.stream(frames_view[:n], LEVELS, out=out_view[:n])

    e2e_run(2)
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record(stream)
    e2e_run(e2e_steps)
    f1.record(stream)
    barrier()
    e2e_ms = f0.elapsed_time(f1)
    # what plain pinned copies of the same bytes reach with every rank copying at once (the ceiling of e2e at this N)
    ceil_ms = copy_ceiling(dev, h * w * 4, (LEVELS + 1) * h * w * 4, barrier)

    # the call users make: wow(host frame) -> host reconstruction (64 MiB in, 64 MiB out per frame), 3-stream pipeline
    wow_out = torch.empty((h, w), dtype=torch.float32).pin_memory()
    wow_in = host_in.abs().mul_(50).pin_memory()
    wow_frames = wow_in.unsqueeze(0).expand(e2e_steps, h, w)
    wow_view = wow_out.unsqueeze(0).expand(e2e_steps, h, w)
    wb.wow_stream(wow_frames[:2], out=wow_view[:2])
    barrier()
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g0.record(stream)
    wb.wow_stream(wow_frames, out=wow_view)
    g1.record(stream)
    barrier()
    e2e_wow_ms = g0.elapsed_time(g1)
    ceil_wow_ms = copy_ceiling(dev, h * w * 4, h * w * 4, barrier)  # one frame each way, both directions at once

    times = torch.tensor([elapsed_ms, e2e_ms, ceil_ms, e2e_wow_ms, ceil_wow_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    elapsed_ms, e2e_ms, ceil_ms, e2e_wow_ms, ceil_wow_ms = times.tolist()

    units_per_step = h * w * LEVELS / 1e6  # Mpixel*scales
    value = units_per_step * args.steps * world / (elapsed_ms / 1e3)
    e2e_value = units_per_step * e2e_steps * world / (e2e_ms / 1e3)
    peak, peak_src = measured_peaks()

    line = None
    if rank == 0:
        launch_ms = elapsed_ms / (args.steps * LEVELS)
        algo_bytes = 3 * 4 * h * w  # read c_s, write c_{s+1}, write w_s
        achieved = algo_bytes / (launch_ms / 1e3) / 1e9
        step_bytes = h * w * 4 + (LEVELS + 1) * h * w * 4
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": warmup, "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": dict(CONFIG),
            "detail": {"kernel": "atrous_rows_lean_kernel<5> (TMA row pipeline, packed fp32x2, PDL)",
                       "e2e_steps": e2e_steps, "numa_cpus_bound": numa_cpus},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": ncu_traffic(), "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": algo_bytes, "launch_ms": launch_ms},
            "cpu_baseline": None,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h * w * 4,
                    "d2h_bytes_per_step": (LEVELS + 1) * h * w * 4, "ms_per_step": e2e_ms / e2e_steps,
                    "api": "AtrousTransform.stream(pinned host frames) -> pinned host planes",
                    "gbs_per_gpu": step_bytes / (e2e_ms / e2e_steps) / 1e6,
                    "plain_copy_ms_per_step": ceil_ms, "plain_copy_gbs_per_gpu": step_bytes / ceil_ms / 1e6,
                    "frac_of_plain_copy": ceil_ms / (e2e_ms / e2e_steps)},
            "e2e_wow": {"frames_per_s": world * e2e_steps / (e2e_wow_ms / 1e3), "ms_per_frame": e2e_wow_ms / e2e_steps,
                        "h2d_bytes_per_step": h * w * 4, "d2h_bytes_per_step": h * w * 4,
                        "plain_copy_ms_per_step": ceil_wow_ms, "frac_of_plain_copy": ceil_wow_ms / (e2e_wow_ms / e2e_steps),
                        "api": "wow_stream(pinned host frames) -> pinned host reconstructions (wow() per frame)"},
            "gpu_launches": args.steps * LEVELS,
            "clocks": clocks,
        }

    # Everything below only ADDS keys.  A watchdog prints the line as it stands if an extra stalls (a collective that
    # never completes must not cost the headline number).
    done = threading.Event()

    def emit(extra_error=None):
        if done.is_set():
            return
        done.set()
        if rank == 0:
            if extra_error:
                line["extras_error"] = extra_error
            print(json.dumps(line), flush=True)

    def watchdog():
        if not done.wait(args.extras_timeout):
            emit(f"extras did not finish within {args.extras_timeout} s")
            os._exit(0)

    threading.Thread(target=watchdog, daemon=True).start()
    err = None
    try:
        # ---- WOW frames/s (BASELINE.json configs[2]), device-resident, rank 0 reports its own GPU ------------------
        if rank == 0 and not args.no_wow:
            solar = solar_like_device(N_SIDE, torch.float32, dev)
            line["wow"] = time_wow(wb, solar, 30, peak)
            line["wow_bilateral"] = time_wow(wb, solar, 15, peak, bilateral=1, denoise_coefficients=[5, 2])
            line["wow"]["call"] = "wow(4096x4096 fp32 solar-like)"
            line["wow_bilateral"]["call"] = "wow(4096x4096 fp32 solar-like, bilateral=1, denoise_coefficients=[5, 2])"
            line["wow_bilateral"]["bound"] = ("instruction issue + MUFU pipe, not HBM: the bilateral scale kernel needs 162 packed "
                                              "fp32x2 operations (two issue cycles each) and 52 MUFU per 64 pixels; its arithmetic "
                                              "alone replayed on the same SM (tools/k2mimic.cu) takes 114 us per 4096^2 scale, "
                                              "the kernel 135-156 us, against 31 us of HBM time for its 3 planes")
            solar64 = solar.to(torch.float64)
            line["wow_f64"] = time_wow(wb, solar64, 10, peak)
            line["wow_bilateral_f64"] = time_wow(wb, solar64, 4, peak, bilateral=1, denoise_coefficients=[5, 2])
            line["wow_f64"]["call"] = "wow(4096x4096 fp64 solar-like)"
            line["wow_bilateral_f64"]["call"] = "wow(4096x4096 fp64 solar-like, bilateral=1, denoise_coefficients=[5, 2])"
            del solar64
            # BASELINE.json configs[3] flavour: a stack of frames, one launch per scale for the whole stack (wow_batch)
            nb = 8
            stack = solar.unsqueeze(0).repeat(nb, 1, 1)
            stack += torch.sqrt(stack.clamp(min=1)) * 0.1 * torch.randn(stack.shape, device=dev)
            for _ in range(2):
                _, pl, _ = wb.wow_batch(stack)
            levels_b = pl.shape[1] - 1
            del pl
            torch.cuda.synchronize(dev)
            b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            b0.record()
            for _ in range(5):
                wb.wow_batch(stack)
            b1.record()
            torch.cuda.synchronize(dev)
            ms_b = b0.elapsed_time(b1) / 5 / nb
            algo_b = (5 * levels_b + 3) * 4 * h * w
            line["wow_batch"] = {"frames_per_s": 1e3 / ms_b, "ms_per_frame": ms_b, "scales": levels_b,
                                 "frames_per_launch": nb, "algorithmic_bytes_per_frame": algo_b,
                                 "achieved_gbs": algo_b / ms_b / 1e6, "frac_of_hbm_peak": algo_b / ms_b / 1e6 / peak,
                                 "call": "wow_batch(8 x 4096x4096 fp32 solar-like)"}
            del stack, solar
            torch.cuda.empty_cache()
        if world > 1 and not args.no_extras:
            del planes, scratch, img
            torch.cuda.empty_cache()
            extras = multi_gpu_extras(args, wb, dist, dev, rank, world, peak)
            if rank == 0:
                line.update(extras)
        # the CPU baseline is timed on rank 0 at N = 1 only (the contract); multi-GPU lines carry null
        if rank == 0 and world == 1:
            os.sched_setaffinity(0, all_cpus)  # the CPU baseline may use every host core again
            cpu_val, cpu_s, backend, threads = cpu_reference_rate(N_SIDE, LEVELS)
            line["cpu_baseline"] = {"value": cpu_val, "unit": UNIT, "cores": threads, "kind": "port",
                                    "sample": f"one full {N_SIDE}x{N_SIDE} fp32 frame, {LEVELS} scales, {cpu_s:.2f} s, "
                                              f"oracle port backend={backend} ({os.cpu_count()} host cpus)"}
    except Exception as exc:  # an extra must never cost the headline line
        err = f"{type(exc).__name__}: {exc}"[:400]
    emit(err)
    if world > 1:
        try:
            dist.destroy_process_group()
        except Exception:
            pass


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-wow", action="store_true", help="skip the extra WOW frames/s measurements")
    ap.add_argument("--no-extras", action="store_true", help="N > 1: skip the cfg4 / cfg5 (banded) keys")
    ap.add_argument("--extras-timeout", type=float, default=300.0,
                    help="seconds after which the line is printed without the extra keys that have not finished")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write a fixed sample of the last step's planes to DIR/planes_sample.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
