"""Row-band sharded cascade on N GPUs vs the same cascade on one GPU: must be BIT-IDENTICAL.

    torchrun --nproc-per-node N --master-addr 127.0.0.1 --master-port 29511 tools/check_banded.py [--side 8192 --levels 10]

Every rank builds the same seeded image, transforms its own band with BandedTransform (NCCL halo exchange per scale),
and compares against the rows of the unsharded transform computed locally.  Also reports timing (max over ranks).
"""
import argparse
import json
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import wavelets_b200 as wb  # noqa: E402
from wavelets_b200.sharded import BandedTransform, band_range  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--side", type=int, default=8192)
    ap.add_argument("--width", type=int, default=0)
    ap.add_argument("--levels", type=int, default=10)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--no-check", action="store_true", help="skip the unsharded comparison (image too large for one GPU)")
    ap.add_argument("--quick", action="store_true", help="B3spline fp32 only")
    ap.add_argument("--modes", default="nccl,p2p,push",
                    help="halo transport: nccl (send/recv exchange), p2p (in-kernel peer reads), push (in-kernel peer writes)")
    ap.add_argument("--out", default="", help="also write the JSON summary to this file (rank 0)")
    args = ap.parse_args()
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    h, w = args.side, (args.width or args.side)
    y0, y1 = band_range(h, rank, world)
    ok = True
    results = {}
    modes = [m for m in args.modes.split(",") if m]
    cases = [(wb.B3spline, torch.float32)] if args.quick else [
        (sf, dt) for sf in (wb.B3spline, wb.Triangle) for dt in (torch.float32, torch.float64)]
    for sf, dt in cases:
        if True:
            gen = torch.Generator(device=dev).manual_seed(7)
            if args.no_check:
                # every rank generates only its band (seeded per rank)
                gen.manual_seed(7 + rank)
                band = torch.randn((y1 - y0, w), generator=gen, device=dev, dtype=torch.float32).to(dt)
            else:
                img = torch.randn((h, w), generator=gen, device=dev, dtype=torch.float32).to(dt)
                band = img[y0:y1].contiguous()
            full = None if args.no_check else wb.AtrousTransform(sf)(img, args.levels).data
            for mode in modes:
                bt = BandedTransform(sf, poison=True, p2p=(mode == "p2p"), push=(mode == "push"))
                planes = bt(band, args.levels, h)
                torch.cuda.synchronize()
                if full is not None:
                    same = torch.equal(planes, full[:, y0:y1])
                    flag = torch.tensor([1 if same else 0], device=dev)
                    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
                    ok = ok and bool(flag.item())
                    if rank == 0:
                        print(f"{sf.__name__:9s} {str(dt):14s} {mode:5s} banded == unsharded on all ranks: "
                              f"{bool(flag.item())}", flush=True)
                del planes
                # timing of the sharded cascade (device time, max over ranks)
                bt = BandedTransform(sf, p2p=(mode == "p2p"), push=(mode == "push"))
                for _ in range(2):
                    bt(band, args.levels, h)
                dist.barrier(); torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(args.reps):
                    bt(band, args.levels, h)
                e1.record()
                dist.barrier(); torch.cuda.synchronize()
                t = torch.tensor([e0.elapsed_time(e1) / args.reps], device=dev, dtype=torch.float64)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                results[f"{sf.__name__}_{str(dt).split('.')[-1]}_{mode}"] = {
                    "ms": t.item(), "mpx_scales_per_s": h * w * args.levels / t.item() / 1e3}
                del bt
            if full is not None:
                del full, img
            del band
            torch.cuda.empty_cache()
    # ---- WOW on bands (two halo exchanges per scale + all-gather of the residual moments) vs the unsharded two-pass wow
    if not args.no_check and not args.quick:
        from wavelets_b200.sharded import BandedWow
        for dt in (torch.float32, torch.float64):
            gen = torch.Generator(device=dev).manual_seed(11)
            img = (torch.randn((h, w), generator=gen, device=dev, dtype=torch.float32) * 5 + 40).to(dt)
            # noise given for float32; float64 estimates it (distributed exact MAD of the raw w_0)
            kw = dict(weights=[1.5, 1.2], denoise_coefficients=[4, 2])
            if dt == torch.float32:
                kw["noise"] = 1.5
            recon_b, planes_b = BandedWow(wb.B3spline, poison=True)(img[y0:y1].contiguous(), h,
                                                                    n_scales=min(args.levels, 6), **kw)
            L = planes_b.shape[0] - 1
            # two-pass reference: wow() of the unsharded coefficients whitens every raw plane with K3
            co = wb.AtrousTransform(wb.B3spline)(img, L)
            co.noise = kw.pop("noise", None)
            recon, co = wb.wow(co, **kw)
            same = torch.equal(planes_b[:L], co.data[:L, y0:y1])
            tol = 1e-5 if dt == torch.float32 else 1e-12
            close = ((recon_b - recon[y0:y1]).abs().max() <= tol * recon.abs().max()) and \
                    ((planes_b[L] - co.data[L, y0:y1]).abs().max() <= tol * co.data[L].abs().max())
            flag = torch.tensor([1 if (same and bool(close)) else 0], device=dev)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            ok = ok and bool(flag.item())
            if rank == 0:
                print(f"{str(dt):14s} banded wow == unsharded two-pass wow on all ranks: {bool(flag.item())}", flush=True)
    if rank == 0:
        line = json.dumps({"check": "banded_vs_unsharded", "n_gpus": world, "side": [h, w], "levels": args.levels,
                           "bit_identical": ok if not args.no_check else None, "timing": results})
        print(line, flush=True)
        if args.out:
            with open(args.out, "w") as fh:
                fh.write(line + "\n")
    dist.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
