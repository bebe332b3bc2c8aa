"""Every kernel route of one scale against the float64 oracle, at every dilation the single-reflection limit allows.

The dispatchers (dispatch in atrous_scale.cu, plan_wow / launch_wow_h in wow_scale.cu) pick a different kernel on each
side of a handful of row widths: the generic gather kernel, the row kernel, the lean K1 on 16 KiB / 8 KiB / 24 KiB
(column strip) ring slots, with or without paired columns, and the generic / 512-thread / 256-thread fused WOW kernels.
The widths below sit on both sides of every boundary; W % 8 == 4 gives an odd vector count, so the second vector of the
last thread is masked.  Heights of 1, 2 and 5 rows reflect many times in y; 33 and 300 rows split the chains into
segments at the small dilations.

Every input and output lives inside a larger buffer (row pitch > W, gap rows between frames, a different pitch per
output) whose bytes outside the frames hold a NaN bit pattern: a store outside the logical region, or a write to an
input, is caught bit for bit, and a pixel that is never written stays NaN and fails the oracle comparison.

The route-plan test at the bottom needs only the built library (no device): it rehearses the case list on any machine."""
import hashlib
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch
from scipy.special import erf

from oracle import atrous_oracle as orc
from tests.conftest import ROOT
from tests.test_wide_parity_gpu import report, smooth_field

WB_F32, WB_F64, WB_ENOT_FUSABLE = 0, 1, -7
TAPS = {"b3spline": 5, "triangle": 3}
DCODE = {np.float32: WB_F32, np.float64: WB_F64}
SCALING = ("b3spline", "triangle")

# tolerances of tests/test_wide_parity_gpu.py: K1 c / w, whitened planes (K3 and fused), K2 c / w.  The whitened planes
# are compared with the float64 whitening of the raw plane the kernel whitened: the oracle's w_s rounded to the dtype
# (K3), or x - c_{s+1} with the kernel's own c_{s+1} (fused; c_{s+1} itself is checked against the oracle).  Against the
# oracle's float64 w_s, w / sqrt(S[w^2]) would amplify the unavoidable rounding of the stored c_{s+1} wherever the local
# power is small (Triangle at d = W on one row: S[w^2] = w^2, an error of 0.5 ulp(c) / |w|) and measure that instead of
# the kernel.  For the same reason the hard-threshold masks must agree exactly: both sides threshold the same w_s.
TOL = {np.float32: dict(c=1e-6, w=5e-6, white=1e-5, k2c=1e-6, k2w=1e-5),
       np.float64: dict(c=1e-14, w=1e-13, white=1e-12, k2c=1e-13, k2w=1e-11)}
SIGMA, SIGMA_E, WEIGHT, NOISE = 2.0, 0.4, 1.5, 0.9
FRAME_NOISE = (0.6, 0.9, 1.3)  # per-frame device noise of the batched launches

# (width, heights) per dtype; comments: K1 route / fused WOW route
FP32_CASES = [
    (510, (3, 33)),     # W % 4 != 0: generic gather kernels / declined
    (508, (2, 33)),     # row kernel / generic fused kernel
    (512, (1, 300)),
    (516, (5, 33)),     # row kernel / 256-thread fused kernel
    (1020, (2, 33)),
    (1024, (1, 300)),
    (1028, (5, 33)),    # lean K1 on 8 KiB slots / 256-thread fused kernel
    (1500, (2, 33)),
    (2044, (5, 33)),
    (2048, (1, 300)),   # Triangle reaches d = W on the 256-thread fused kernel
    (2052, (2, 33)),    # lean K1 on 16 KiB slots / 512-thread fused kernel
    (4092, (5, 33)),
    (4096, (1, 33)),    # Triangle reaches d = W on the 512-thread fused kernel
    (4100, (2, 33)),    # lean K1 column strips (row kernel strips at the deep scales) / fused declined
    (6000, (5, 33)),
]
FP64_CASES = [
    (509, (3, 33)),     # odd width: generic gather kernels / declined
    (508, (2, 33)),     # row kernel / generic fused kernel
    (1024, (1, 300)),
    (2044, (5, 33)),    # row kernel, lean 24 KiB-slot kernel with paired columns / generic fused kernel
    (2048, (2, 33)),
    (2052, (1, 33)),    # column strips / fused declined
]
CASES = [(np.float32, w, hs) for w, hs in FP32_CASES] + [(np.float64, w, hs) for w, hs in FP64_CASES]


def scales_of(sf, w):
    """Every scale whose dilation keeps the taps within one reflection in x: c 2^s <= W."""
    c = TAPS[sf] // 2
    return [s for s in range(31) if c * 2 ** s <= w]


def fused_takes(dt, w):
    """The fused kernel stages whole rows: vector-multiple widths up to one 16 KiB row."""
    es = np.dtype(dt).itemsize
    return w % (16 // es) == 0 and w * es <= 16384


def k1_fast_path(dt, w):
    v = 16 // np.dtype(dt).itemsize
    return w % v == 0 and w >= 8 * v


# ---------------------------------------------------------------------------------------------------------------------
# Guard-banded device buffers
# ---------------------------------------------------------------------------------------------------------------------
SENTINEL = {np.float32: (torch.int32, 0x7FA5A5A5), np.float64: (torch.int64, 0x7FF5A5A5A5A5A5A5)}  # NaN payloads


class Guarded:
    """`b` frames of h x w inside a larger device buffer: a guard row and a vector before frame 0, rows of w + pad
    vectors, `gap` rows between frames, a guard row after the last.  Every element outside the frames (and, until
    written, inside them) holds a NaN bit pattern."""

    def __init__(self, dt, shape, pad=1, gap=1, lead=1, data=None):
        self.dt = dt
        self.b, self.h, self.w = shape
        v = 16 // np.dtype(dt).itemsize
        self.pitch = self.w + pad * v
        self.bstride = (self.h + gap) * self.pitch
        lead_el = lead * self.pitch + v
        n = lead_el + self.b * self.bstride + self.pitch
        self.int_t, self.sentinel = SENTINEL[dt]
        self.flat = torch.empty(n, dtype=getattr(torch, np.dtype(dt).name), device="cuda")
        self.flat.view(self.int_t).fill_(self.sentinel)
        self.view = torch.as_strided(self.flat, (self.b, self.h, self.w), (self.bstride, self.pitch, 1), lead_el)
        self.guard = np.ones(n, dtype=bool)
        self.guard[lead_el:lead_el + self.b * self.bstride].reshape(self.b, self.h + gap, self.pitch)[:, :self.h, :self.w] = False
        self.before = None
        if data is not None:
            self.view.copy_(torch.from_numpy(np.ascontiguousarray(data)))
            self.before = self.bits()

    @property
    def ptr(self):
        return self.view.data_ptr()

    def bits(self):
        return self.flat.view(self.int_t).cpu().numpy()

    def get(self):
        return self.view.contiguous().cpu().numpy()

    def _where(self, idx):
        # flat index -> (frame, row, column) relative to frame 0's first element (negative: before it)
        off = int(idx) - (self.view.storage_offset())
        f, rem = divmod(off, self.bstride)
        y, x = divmod(rem, self.pitch)
        return f, y, x

    def check_guard(self, what):
        bits = self.bits()
        bad = np.nonzero(self.guard & (bits != self.sentinel))[0]
        assert bad.size == 0, f"{what}: {bad.size} store(s) outside the frames, first at (frame, row, col) {self._where(bad[0])}"

    def check_unchanged(self, what):
        bits = self.bits()
        bad = np.nonzero(bits != self.before)[0]
        assert bad.size == 0, f"{what}: input written, {bad.size} element(s), first at {self._where(bad[0])}"

    def check_untouched(self, what):
        bits = self.bits()
        assert (bits == self.sentinel).all(), f"{what}: written although the call was declined"


def _opt(g, attr):
    return getattr(g, attr) if g is not None else 0


def _stream():
    return torch.cuda.current_stream().cuda_stream


def launch_k1(lib, src, oc, ow, s, sf):
    return lib.wb_atrous_scale(src.ptr, oc.ptr if oc else None, ow.ptr if ow else None, src.b, src.h, src.w,
                               src.pitch, src.bstride, _opt(oc, "pitch"), _opt(oc, "bstride"), _opt(ow, "pitch"),
                               _opt(ow, "bstride"), s, TAPS[sf], DCODE[src.dt], _stream())


def launch_k2(lib, src, oc, ow, s, sf, vf):
    return lib.wb_atrous_scale_bilateral(src.ptr, oc.ptr, ow.ptr, src.b, src.h, src.w, src.pitch, src.bstride,
                                         oc.pitch, oc.bstride, ow.pitch, ow.bstride, s, TAPS[sf], DCODE[src.dt], vf,
                                         _stream())


def launch_k3(lib, win, out, s, sf, mode, noise_host, noise_dev):
    return lib.wb_wow_whiten_scale(win.ptr, out.ptr, win.b, win.h, win.w, win.pitch, win.bstride, out.pitch,
                                   out.bstride, s, TAPS[sf], DCODE[win.dt], mode, SIGMA, SIGMA_E, noise_host, noise_dev,
                                   WEIGHT, _stream())


def launch_fused(lib, src, oc, ow, s, sf, mode, noise_host, noise_dev):
    return lib.wb_wow_scale(src.ptr, oc.ptr, ow.ptr, src.b, src.h, src.w, src.pitch, src.bstride, oc.pitch,
                            oc.bstride, ow.pitch, ow.bstride, s, TAPS[sf], DCODE[src.dt], mode, SIGMA, SIGMA_E,
                            noise_host, noise_dev, WEIGHT, _stream())


# ---------------------------------------------------------------------------------------------------------------------
# Oracle and comparison
# ---------------------------------------------------------------------------------------------------------------------
def ref_smooth(frames64, sf, s):
    return np.stack([orc.smooth(f, sf, s, backend="numpy") for f in frames64])


def ref_bilateral(f64, sf, s, var_factor):
    """c_{s+1} of one bilateral scale (watroo/wavelets.py:24-32, :74-105, as orc.local_variance + orc.bilateral_smooth)
    evaluated in extended precision, with the local variance in its centred form S[(x - S[x])^2], which equals
    S[x^2] - S[x]^2 without the cancellation: where a pixel and the taps it reaches nearly agree (Triangle at d = W on
    a two-row frame: var / S[x^2] = 2e-10), the float64 difference of the two smooths is off by 1e-6 relative and moves
    c_{s+1} by 6e-13 -- the reference would then measure its own rounding, not the kernel's.  The symmetric border is
    an index reflection instead of np.pad (no padded copy c d rows and columns wider on each side: 800 MB for one
    4096-column row at d = 4096)."""
    x = f64.astype(np.longdouble)
    taps = np.asarray(orc.TAPS[sf], dtype=np.longdouble)
    k2d = np.outer(taps, taps)
    n, c, d = len(taps), len(taps) // 2, 2 ** s
    h, w = x.shape
    ys, xs = np.arange(h), np.arange(w)
    ry = [orc.reflect_index(ys + (i - c) * d, h) for i in range(n)]
    rx = [orc.reflect_index(xs + (j - c) * d, w) for j in range(n)]

    def tap(i, j):
        return x[ry[i]][:, rx[j]]

    mean = sum(k2d[i, j] * tap(i, j) for i in range(n) for j in range(n))
    variance = sum(k2d[i, j] * (tap(i, j) - mean) ** 2 for i in range(n) for j in range(n))
    variance[variance <= 0] = 1e-20
    variance *= var_factor
    out = k2d[c, c] * x
    norm = np.full_like(x, k2d[c, c])
    for i in range(n):
        for j in range(n):
            if i == c and j == c:
                continue
            shifted = tap(i, j)
            weight = k2d[i, j] * np.exp(-((x - shifted) ** 2) / variance / 2)
            norm += weight
            out += shifted * weight
    return (out / norm).astype(np.float64)


def ref_whiten(w64, power, mode, noise):
    """w * significance(w) * weight / sqrt(S[w^2]) in float64, one noise value per frame."""
    p = np.where(power <= 0, 1e-15, power)
    thr = (SIGMA * np.asarray(noise, dtype=np.float64)[:, None, None]) * SIGMA_E
    sig = 1.0 if mode == 0 else (erf(np.abs(w64 / thr)) if mode == 1 else (np.abs(w64) > thr))
    return w64 * sig * (WEIGHT / np.sqrt(p))


class Parity:
    """Worst E_max per route of one test (max norm per plane, SURVEY.md 8(d)) and, for the A/B switch runs, the sha1 of
    every output."""

    def __init__(self):
        self.worst = {}
        self.digests = None  # dict: output key -> sha1 of its bytes (A/B switch runs)

    def close(self, route, got, want, tol, ctx):
        for f in range(len(want)):
            e = orc.emax(got[f], want[f])
            assert e <= tol, (route, ctx, f"frame {f}", e)  # (a NaN -- a pixel never written -- fails too)
            self.worst[route] = max(self.worst.get(route, 0.0), e)

    def digest(self, key, g):
        if self.digests is not None:
            self.digests[key] = hashlib.sha1(g.get().tobytes()).hexdigest()

    def summary(self):
        return ";  ".join(f"{k} {v:.2e}" for k, v in sorted(self.worst.items()))


def check_scale(lib, par, img, s, sf, modes=(0, 1, 2), frame_noise=None, bilateral=False, null_forms=False):
    """K1, K3 (on the oracle's raw plane rounded to the dtype) and the fused scale on the frames `img` (b, h, w), plus
    K2 when `bilateral`, all inside guard-banded buffers, each output against the float64 oracle.  `frame_noise`: None ->
    the host scalar NOISE; else one value per frame, read by the kernels from a device array (the host scalar passed
    beside it is a decoy)."""
    dt = img.dtype.type
    b, h, w = img.shape
    tol = TOL[dt]
    ctx = f"{np.dtype(dt).name} {sf} b{b} {h}x{w} s{s}"
    key = f"{np.dtype(dt).name}/{sf}/{b}x{h}x{w}/s{s}"
    taps = TAPS[sf]
    img64 = img.astype(np.float64)
    c64 = ref_smooth(img64, sf, s)
    w64 = img64 - c64
    if frame_noise is None:
        noise, host, dev_t = [NOISE] * b, NOISE, None
    else:
        noise, host = list(frame_noise), 50.0
        dev_t = torch.tensor(noise, dtype=torch.float64, device="cuda")
    dev = dev_t.data_ptr() if dev_t is not None else None
    src = Guarded(dt, img.shape, pad=1, gap=1, data=img)
    shape = img.shape

    # K1 (+ the smooth-only and detail-only forms)
    oc, ow = Guarded(dt, shape, pad=2, gap=2), Guarded(dt, shape, pad=3, gap=1, lead=2)
    assert launch_k1(lib, src, oc, ow, s, sf) == 0, ctx
    oc.check_guard(f"K1 c {ctx}")
    ow.check_guard(f"K1 w {ctx}")
    src.check_unchanged(f"K1 {ctx}")
    got_c, got_w = oc.get(), ow.get()
    par.close("K1 c", got_c, c64, tol["c"], ctx)
    par.close("K1 w", got_w, w64, tol["w"], ctx)
    par.digest(f"{key}/k1c", oc)
    par.digest(f"{key}/k1w", ow)
    if null_forms:
        only_c = Guarded(dt, shape, pad=1, gap=3)
        assert launch_k1(lib, src, only_c, None, s, sf) == 0, ctx
        only_c.check_guard(f"K1 c (out_w NULL) {ctx}")
        assert np.array_equal(only_c.get(), got_c), ctx
        only_w = Guarded(dt, shape, pad=4, gap=1)
        assert launch_k1(lib, src, None, only_w, s, sf) == 0, ctx
        only_w.check_guard(f"K1 w (out_c NULL) {ctx}")
        assert np.array_equal(only_w.get(), got_w), ctx
        src.check_unchanged(f"K1 NULL forms {ctx}")

    # K3 on the oracle's raw plane, rounded to the plane dtype
    wr = w64.astype(dt)
    wr64 = wr.astype(np.float64)
    p_r = ref_smooth(wr64 * wr64, sf, s)
    win = Guarded(dt, shape, pad=2, gap=1, data=wr)
    for mode in modes:
        out = Guarded(dt, shape, pad=1, gap=3)
        assert launch_k3(lib, win, out, s, sf, mode, host, dev) == 0, (ctx, mode)
        out.check_guard(f"K3 mode {mode} {ctx}")
        win.check_unchanged(f"K3 mode {mode} {ctx}")
        par.close(f"K3 mode {mode}", out.get(), ref_whiten(wr64, p_r, mode, noise), tol["white"], (ctx, mode))
        par.digest(f"{key}/k3m{mode}", out)

    # fused K1 + K3
    takes = fused_takes(dt, w)
    oc, ow = Guarded(dt, shape, pad=3, gap=2), Guarded(dt, shape, pad=1, gap=1, lead=3)
    assert lib.wb_wow_scale_path(b, h, w, src.pitch, oc.pitch, ow.pitch, s, taps, DCODE[dt], src.ptr, oc.ptr,
                                 ow.ptr) == int(takes), ctx
    for mode in modes:
        oc, ow = Guarded(dt, shape, pad=3, gap=2), Guarded(dt, shape, pad=1, gap=1, lead=3)
        rc = launch_fused(lib, src, oc, ow, s, sf, mode, host, dev)
        if not takes:
            assert rc == WB_ENOT_FUSABLE, (ctx, rc)
            oc.check_untouched(f"fused c {ctx}")
            ow.check_untouched(f"fused w {ctx}")
            continue
        assert rc == 0, (ctx, mode, rc)
        oc.check_guard(f"fused c mode {mode} {ctx}")
        ow.check_guard(f"fused w mode {mode} {ctx}")
        src.check_unchanged(f"fused mode {mode} {ctx}")
        got_c = oc.get()
        par.close("fused c", got_c, c64, tol["c"], (ctx, mode))
        wk = (img - got_c).astype(np.float64)  # the raw plane the kernel whitened: x - c_{s+1} in the plane dtype
        par.close(f"fused mode {mode}", ow.get(), ref_whiten(wk, ref_smooth(wk * wk, sf, s), mode, noise),
                  tol["white"], (ctx, mode))
        par.digest(f"{key}/fc{mode}", oc)
        par.digest(f"{key}/fw{mode}", ow)

    # K2 (bilateral smooth)
    if bilateral:
        vf = 2.25 * (s + 1)
        k2c = np.stack([ref_bilateral(f, sf, s, vf) for f in img64])
        oc, ow = Guarded(dt, shape, pad=2, gap=1), Guarded(dt, shape, pad=1, gap=2)
        assert launch_k2(lib, src, oc, ow, s, sf, vf) == 0, ctx
        oc.check_guard(f"K2 c {ctx}")
        ow.check_guard(f"K2 w {ctx}")
        src.check_unchanged(f"K2 {ctx}")
        par.close("K2 c", oc.get(), k2c, tol["k2c"], ctx)
        par.close("K2 w", ow.get(), img64 - k2c, tol["k2w"], ctx)
        par.digest(f"{key}/k2c", oc)
        par.digest(f"{key}/k2w", ow)


def _gpu_lib():
    from wavelets_b200 import _lib
    return _lib.load(require_cuda=True)


def _frames(b, h, w, dt, seed):
    return np.stack([smooth_field(h, w, seed + 101 * f, dt) for f in range(b)])


def _case_id(case):
    dt, w, hs = case
    return f"{np.dtype(dt).name}-{w}"


# ---------------------------------------------------------------------------------------------------------------------
# 1. every route, every dilation
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("sf", SCALING)
@pytest.mark.parametrize("case", CASES, ids=_case_id)
def test_every_route_every_dilation_vs_oracle(case, sf):
    """K1, K3 and the fused scale at every dilation up to the single-reflection limit (d = W for Triangle on power-of-two
    widths), all three significance modes, single frames in pitched buffers; K2 at the deepest dilation."""
    dt, w, heights = case
    lib = _gpu_lib()
    par = Parity()
    scales = scales_of(sf, w)
    for h in heights:
        img = _frames(1, h, w, dt, 17 + w + h)
        for s in scales:
            check_scale(lib, par, img, s, sf, bilateral=(s == scales[-1]))
    report(f"route parity {np.dtype(dt).name} {sf:8s} W={w} H={heights} s=0..{scales[-1]}: {par.summary()}")


@pytest.mark.gpu
@pytest.mark.parametrize("dt", [np.float32, np.float64])
@pytest.mark.parametrize("sf", SCALING)
def test_row_kernel_one_vector_per_thread_vs_oracle(sf, dt):
    """The row kernel with one column vector per thread (the geometry override of wb_tune_k1, ng = 1) for K1 and K3."""
    lib = _gpu_lib()
    par = Parity()
    w = 1024
    nt = w // (16 // np.dtype(dt).itemsize)
    nt = min(nt, 512)
    img = _frames(1, 45, w, dt, 5)
    try:
        for s in scales_of(sf, w):
            assert lib.wb_tune_k1(s, nt, 1, 8, 0) == 0
            check_scale(lib, par, img, s, sf, modes=(0, 1, 2))
    finally:
        for s in range(32):
            lib.wb_tune_k1(s, 0, 0, 0, 0)
    report(f"row kernel ng=1 {np.dtype(dt).name} {sf:8s} 45x{w}: {par.summary()}")


# ---------------------------------------------------------------------------------------------------------------------
# 2. batches of different frames, per-frame device noise, both NULL output forms of K1
# ---------------------------------------------------------------------------------------------------------------------
BATCH_WIDTHS = {np.float32: (508, 1020, 1500, 2048, 4092, 4096, 6000), np.float64: (508, 1024, 2048, 2052)}


@pytest.mark.gpu
@pytest.mark.parametrize("dt", [np.float32, np.float64])
@pytest.mark.parametrize("sf", SCALING)
def test_batched_frames_per_frame_noise_vs_oracle(sf, dt):
    """Three different frames per launch in guard-banded buffers, per-frame noise read from the device: each frame is
    checked against the oracle with its own noise, so a frame-indexing error common to all routes cannot pass."""
    lib = _gpu_lib()
    par = Parity()
    for w in BATCH_WIDTHS[dt]:
        img = _frames(3, 37, w, dt, 300 + w)
        sc = scales_of(sf, w)
        for s in sorted({0, 1, 2, 3, 5, sc[-2], sc[-1]}):
            check_scale(lib, par, img, s, sf, frame_noise=FRAME_NOISE, null_forms=True,
                        bilateral=s in (0, sc[-1]))
    report(f"route parity batch 3 {np.dtype(dt).name} {sf:8s} W={BATCH_WIDTHS[dt]}: {par.summary()}")


# ---------------------------------------------------------------------------------------------------------------------
# 3. route coverage: the cases above launch every kernel family the dispatchers can pick
# ---------------------------------------------------------------------------------------------------------------------
EXPECTED_FAMILIES = sorted(
    ["atrous_generic_kernel", "atrous_rows_kernel ng=1", "atrous_rows_kernel ng=2",
     "atrous_rows_lean_kernel 16 KiB slots", "atrous_rows_lean_kernel 8 KiB slots", "atrous_rows_lean_kernel strip",
     "atrous_rows_lean_kernel paired", "atrous_rows_lean_kernel OP_WHITEN", "wow_rows_kernel"]
    + [f"wow_rows_lean_kernel {nt} threads {pr} mode {m}" for nt in (512, 256) for pr in ("paired", "unpaired")
       for m in (0, 1, 2)])
_KERNEL_RE = re.compile(r"\b(atrous_generic_kernel|atrous_rows_lean_kernel|atrous_rows_kernel|wow_rows_lean_kernel|"
                        r"wow_rows_kernel)<([^>]*)>")


def kernel_families(name):
    """Families of one demangled kernel name (template arguments as in atrous_scale.cu / wow_scale.cu)."""
    m = _KERNEL_RE.search(name)
    if not m:
        return set()
    kern = m.group(1)
    args = [re.sub(r"\((?:int|bool)\)", "", a).strip() for a in m.group(2).split(",")]
    args = [{"true": "1", "false": "0"}.get(a, a) for a in args]
    if kern == "atrous_generic_kernel" or kern == "wow_rows_kernel":
        return {kern}
    if kern == "atrous_rows_kernel":  # <T, TAPS, DMODE, NG, OP>
        return {f"atrous_rows_kernel ng={args[3]}"}
    if kern == "atrous_rows_lean_kernel":  # <T, TAPS, DMODE, HINTS, OP, MODE, PAIR, UNROLL, RBK>
        rbk = args[8] if len(args) > 8 else "16"
        fams = {"atrous_rows_lean_kernel " + {"16": "16 KiB slots", "8": "8 KiB slots", "24": "strip"}[rbk]}
        if len(args) > 6 and args[6] != "0":
            fams.add("atrous_rows_lean_kernel paired")
        if len(args) > 4 and args[4] == "1":
            fams.add("atrous_rows_lean_kernel OP_WHITEN")
        return fams
    # wow_rows_lean_kernel<TAPS, DMODE, HINTS, MODE, PAIR, DYN, NTK>
    ntk = args[6] if len(args) > 6 else "512"
    pair = len(args) > 4 and args[4] != "0"
    return {f"wow_rows_lean_kernel {ntk} threads {'paired' if pair else 'unpaired'} mode {args[3]}"}


def test_kernel_family_parser():
    assert kernel_families("void wb::atrous_rows_lean_kernel<float, (int)3, (int)0, (bool)1, (int)0, (int)0, (int)1, "
                           "(int)4, (int)8>(wb::ScaleParams)") == {"atrous_rows_lean_kernel 8 KiB slots",
                                                                    "atrous_rows_lean_kernel paired"}
    assert kernel_families("void wb::wow_rows_lean_kernel<5, 0, true, 2, 1, true, 256>(wb::ScaleParams)") == {
        "wow_rows_lean_kernel 256 threads paired mode 2"}
    assert kernel_families("void wb::atrous_rows_kernel<double, 5, 1, 1, 1>(wb::ScaleParams)") == {"atrous_rows_kernel ng=1"}
    assert kernel_families("void wb::atrous_rows_lean_kernel<double, 5, 0, true, 1, 2, 0, 4, 24>(wb::ScaleParams)") == {
        "atrous_rows_lean_kernel strip", "atrous_rows_lean_kernel OP_WHITEN"}
    assert kernel_families("void at::native::vectorized_elementwise_kernel<4, float>()") == set()


@pytest.mark.gpu
def test_route_coverage():
    """Runs the route cases once more (smallest height of each) under torch.profiler and checks that every kernel family
    the dispatchers can pick was launched, so that a planner change cannot move the cases off a kernel unnoticed."""
    from torch.profiler import ProfilerActivity, profile
    lib = _gpu_lib()
    par = Parity()
    seen = {}
    with profile(activities=[ProfilerActivity.CUDA], acc_events=True) as prof:
        for dt, w, heights in CASES:
            for sf in SCALING:
                img = _frames(1, heights[0], w, dt, 23 + w)
                for s in scales_of(sf, w):
                    check_scale(lib, par, img, s, sf)
        img = _frames(1, 9, 1024, np.float32, 3)
        try:
            assert lib.wb_tune_k1(4, 256, 1, 8, 0) == 0
            check_scale(lib, par, img, 4, "b3spline", modes=(1,))
        finally:
            lib.wb_tune_k1(4, 0, 0, 0, 0)
        torch.cuda.synchronize()
    for ev in prof.events():
        for fam in kernel_families(ev.name):
            seen[fam] = seen.get(fam, 0) + 1
    missing = [f for f in EXPECTED_FAMILIES if f not in seen]
    report("route coverage: " + ", ".join(f"{f} x{seen[f]}" for f in sorted(seen)))
    assert not missing, f"kernel families never launched: {missing}"


# ---------------------------------------------------------------------------------------------------------------------
# 4. the A/B environment switches
# ---------------------------------------------------------------------------------------------------------------------
SWITCH_CASES = [(np.float32, 1020), (np.float32, 1500), (np.float32, 2048), (np.float32, 3000), (np.float32, 4096),
                (np.float32, 6000), (np.float64, 1024), (np.float64, 2048), (np.float64, 3000)]
SWITCH_VARS = ("WB_PDL", "WB_L2_HINTS", "WB_L2_HINTS_WOW", "WB_K1_UNROLL", "WB_WOW_DYN", "WB_K1_LEAN", "WB_WOW_LEAN",
               "WB_K1_PAIR", "WB_WOW_PAIR", "WB_K1_LEAN_STRIPS", "WB_WOW_STRIPS", "WB_K2_WINDOW")
# Every switch must give planes bit-identical to the default (measured on a B200 for all of them).  The first eight
# change scheduling, cache hints or loop shape only; the last five run another kernel (generic instead of lean, unpaired
# instead of paired columns, the row kernel instead of lean strips) that performs the same operations in the same order.
SWITCHES = ["WB_PDL=0", "WB_L2_HINTS=0", "WB_L2_HINTS_WOW=0", "WB_L2_HINTS_WOW=1", "WB_L2_HINTS_WOW=2", "WB_K1_UNROLL=8",
            "WB_WOW_DYN=0", "WB_WOW_DYN=1",
            "WB_K1_LEAN=0", "WB_WOW_LEAN=0", "WB_K1_PAIR=0", "WB_WOW_PAIR=0", "WB_K1_LEAN_STRIPS=0"]

_CHILD = """
import json, sys
sys.path.insert(0, {root!r})
from tests.test_route_parity_gpu import run_switch_cases
json.dump(run_switch_cases(), open(sys.argv[1], "w"))
"""


def run_switch_cases():
    """The compact case list of the switch test, in this process (whatever WB_* variables it was started with): every
    output checked against the oracle; returns the sha1 of every output."""
    lib = _gpu_lib()
    par = Parity()
    par.digests = {}
    for dt, w in SWITCH_CASES:
        for sf in SCALING:
            img = _frames(1, 19, w, dt, 71 + w)
            for s in scales_of(sf, w):
                check_scale(lib, par, img, s, sf, bilateral=s in (0, 3))
    return par.digests


@pytest.mark.gpu
def test_ab_switches(tmp_path):
    """Each A/B switch in a fresh process (the library reads them once): every output meets the oracle tolerance and is
    bit-identical to the default run, so that A/B timings compare two ways of computing the same planes."""
    settings = [None] + SWITCHES
    base_env = {k: v for k, v in os.environ.items() if k not in SWITCH_VARS}
    script = _CHILD.format(root=ROOT)
    results, procs = {}, []
    try:
        pending = list(settings)
        while pending or procs:
            while pending and len(procs) < 4:
                setting = pending.pop(0)
                env = dict(base_env)
                if setting:
                    k, v = setting.split("=")
                    env[k] = v
                out = tmp_path / f"{setting or 'default'}.json"
                log = open(tmp_path / f"{setting or 'default'}.log", "w")
                p = subprocess.Popen([sys.executable, "-c", script, str(out)], cwd=ROOT, env=env, stdout=log,
                                     stderr=subprocess.STDOUT)
                procs.append((setting, p, out, log))
            setting, p, out, log = procs[0]
            rc = p.wait(timeout=900)
            procs.pop(0)
            log.close()
            text = open(log.name).read()
            assert rc == 0, f"{setting or 'default'}: child failed (oracle tolerance or launch):\n{text[-4000:]}"
            results[setting] = json.load(open(out))
    finally:
        for _, p, _, log in procs:
            p.kill()
            p.wait()
            log.close()
    base = results[None]
    lines, not_identical = [], []
    for setting in settings[1:]:
        got = results[setting]
        assert got.keys() == base.keys(), setting
        diff = sorted(k for k in base if got[k] != base[k])
        lines.append(f"{setting}: {'bit-identical' if not diff else f'{len(diff)} of {len(base)} outputs differ'}")
        if diff:
            not_identical.append((setting, diff[:6]))
    report(f"A/B switches ({len(base)} outputs each, all within the oracle tolerance): " + "; ".join(lines))
    assert not not_identical, not_identical


# ---------------------------------------------------------------------------------------------------------------------
# host only: the route plan of the case list (needs the built library, no device)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def host_lib():
    from wavelets_b200.build import build_library
    build_library()
    from wavelets_b200 import _lib
    return _lib.load()


def test_route_plan_of_the_case_list(host_lib):
    """wb_atrous_scale_path / wb_wow_scale_path accept the cases as the GPU tests above expect -- at every scale, with
    the pitches of the guard-banded buffers -- so the case list can be rehearsed without a device."""
    import ctypes
    lib = host_lib
    fake = [ctypes.c_void_p(256 * (k + 1)) for k in range(3)]  # 16-byte aligned stand-ins (nothing is launched)
    n_fused = {}
    for dt, w, heights in CASES + [(dt, w, (19,)) for dt, w in SWITCH_CASES]:
        v = 16 // np.dtype(dt).itemsize
        for sf in SCALING:
            for s in scales_of(sf, w):
                for h in heights:
                    for pitch in (w, w + v, w + 3 * v):
                        assert lib.wb_atrous_scale_path(h, w, pitch, pitch, s, TAPS[sf], DCODE[dt], None, None,
                                                        None) == int(k1_fast_path(dt, w)), (dt, w, h, s, sf)
                        for b in (1, 3):
                            got = lib.wb_wow_scale_path(b, h, w, pitch, pitch + v, pitch + 2 * v, s, TAPS[sf],
                                                        DCODE[dt], *fake)
                            assert got == int(fused_takes(dt, w)), (dt, w, h, s, sf, b)
                            n_fused[(np.dtype(dt).name, w, sf, s)] = got
    # the deepest dilations the fused kernels take: d = W on both lean kernels (256 and 512 threads)
    assert n_fused[("float32", 2048, "triangle", 11)] == 1 and n_fused[("float32", 4096, "triangle", 12)] == 1
    assert n_fused[("float64", 2048, "triangle", 11)] == 1
    # one scale beyond the single reflection goes to the generic kernel, the fused kernel declines it
    assert lib.wb_atrous_scale_path(33, 2048, 2048, 2048, 12, 3, WB_F32, None, None, None) == 0
    assert lib.wb_wow_scale_path(1, 33, 2048, 2048, 2048, 2048, 12, 3, WB_F32, *fake) == 0
