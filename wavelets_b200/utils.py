"""Applications on top of the transform: ``denoise`` and ``wow`` (mirror of watroo/utils.py:83-102, :105-219).

Both keep the reference's signatures and quirks (``denoise``'s ``weights`` are the sigma thresholds; ``wow`` returns
``(recon, coefficients)`` with the planes overwritten by their whitened values).  NumPy in -> NumPy out for the image
results; torch tensor in -> torch CUDA tensor out.  ``coefficients.data`` always stays on the device.
"""
from __future__ import annotations

import copy
import ctypes
import numbers
import warnings

import numpy as np
import torch

from . import _lib
from .scaling import B3spline
from .wavelets import (AtrousTransform, Coefficients, _Noise, _frame_layout, abs_median_noise, atrous_scale,
                       bilateral_list, broadcast_noise_map, plane_moments, synthesis, to_device_image)

__all__ = ["denoise", "wow", "wow_batch", "wow_stream", "generalized_anscombe", "enhance", "richardson_lucy"]

_PIPELINE_STREAMS: dict = {}


def _pipeline_streams(device):
    """The (upload, compute, download) streams of the host-frame pipelines, created once per device: the caching
    allocator keeps one pool per stream, so fresh streams per call would start every call with cudaMalloc."""
    key = (device.type, device.index)
    st = _PIPELINE_STREAMS.get(key)
    if st is None:
        st = _PIPELINE_STREAMS[key] = tuple(torch.cuda.Stream(device) for _ in range(3))
    return st


def generalized_anscombe(signal, alpha=1, g=0, sigma=0, inverse=False):
    """Variance-stabilising transform and its algebraic inverse (watroo/wavelets.py:14-21), element-wise on a torch
    tensor (device or host)."""
    if inverse:
        return ((alpha * signal / 2) ** 2 + alpha * g - sigma ** 2 - 3 * alpha / 8) / alpha
    dum = alpha * signal + 3 * alpha ** 2 / 8 + sigma ** 2 - alpha * g
    return 2 * torch.sqrt(torch.clamp(dum, min=0)) / alpha


def _result(t, as_numpy):
    return t.cpu().numpy() if as_numpy else t


def denoise(data, weights, scaling_function=B3spline, noise=None, bilateral=None, soft_threshold=True,
            anscombe=False):
    """Convenience denoiser (watroo/utils.py:83-102).  NB ``weights`` are the sigma thresholds of each scale and
    their count sets the number of scales; the result is the sum of the thresholded planes."""
    img, was_numpy = to_device_image(data, ndim_ok=(1, 2, 3))  # 1-D signals and 3-D volumes: plain cascade only
    if anscombe:
        img = generalized_anscombe(img)
    transform = AtrousTransform(scaling_function, bilateral=bilateral)
    coefficients = transform(img, len(weights))
    coefficients.noise = noise
    coefficients.denoise(weights, soft_threshold=soft_threshold)
    planes = coefficients.data
    out = synthesis(planes if img.ndim == 2 else planes.reshape(planes.shape[0], 1, -1)).reshape(img.shape)
    if anscombe:
        out = generalized_anscombe(out, inverse=True)
    return _result(out, was_numpy)


def _wow_plan(shape, scaling_function, n_scales, weights, denoise_coefficients, bilateral, from_coefficients=None,
              h=0, n_dims=2):
    """Scale-count and per-scale parameter lists of wow() (watroo/utils.py:121-146, :160-170)."""
    n_taps = len(scaling_function.coefficients_1d)
    if from_coefficients is None:
        max_scales = int(np.round(np.log2(min(shape)) - np.log2(n_taps)))
        if n_scales is None:
            n_scales = max_scales if h < 1 else len(denoise_coefficients)  # utils.py:123-124
        elif n_scales > max_scales:
            n_scales = max_scales
    else:
        n_scales = len(from_coefficients) - 1
    table_len = len(scaling_function(n_dims).sigma_e(bilateral=bilateral))
    if len(denoise_coefficients) >= table_len:
        warnings.warn(f"Required number of scales lager then the maximum for scaling function. Using {table_len}.")
        n_scales = table_len
    sigma_bilateral = None if bilateral is None else bilateral_list(bilateral, n_scales)
    wts = copy.copy(list(weights))
    if len(wts) <= n_scales:
        wts.extend([1, ] * (n_scales - len(wts) + 1))
    dns = copy.copy(list(denoise_coefficients))
    if len(dns) < n_scales:
        dns.extend([0, ] * (n_scales - len(dns)))
    if len(dns) == n_scales:
        dns.extend([1, ])
    return n_scales, sigma_bilateral, wts, dns


def _whiten_scale(lib, w_raw, out, s, scaling_function, sig_mode, sigma, sigma_e, nz, weight):
    b, h, w, pitch, bstride = _frame_layout(w_raw)
    _, _, _, o_pitch, o_bstride = _frame_layout(out)
    with torch.cuda.device(w_raw.device):
        _lib.check(lib.wb_wow_whiten_scale(w_raw.data_ptr(), out.data_ptr(), b, h, w, pitch, bstride, o_pitch,
                                           o_bstride, s, scaling_function.taps_code, _lib.dtype_code(w_raw.dtype),
                                           sig_mode, float(sigma), float(sigma_e), nz.host, nz.dev_ptr, float(weight),
                                           _lib.stream_ptr(w_raw.device)))


def _whiten_scale_map(lib, w_raw, out, noise_map, s, scaling_function, soft, sigma, sigma_e, weight):
    """K3 with a per-pixel noise map (wb_wow_whiten_scale_map): ``noise_map`` is (H, W), shared by every frame, or one
    (H, W) map per frame of ``w_raw``."""
    b, h, w, pitch, bstride = _frame_layout(w_raw)
    _, _, _, o_pitch, o_bstride = _frame_layout(out)
    _, _, _, m_pitch, m_bstride = _frame_layout(noise_map)
    with torch.cuda.device(w_raw.device):
        _lib.check(lib.wb_wow_whiten_scale_map(w_raw.data_ptr(), out.data_ptr(), noise_map.data_ptr(), b, h, w, pitch,
                                               bstride, o_pitch, o_bstride, m_pitch, m_bstride, s,
                                               scaling_function.taps_code, _lib.dtype_code(w_raw.dtype),
                                               1 if soft else 0, float(sigma), float(sigma_e), float(weight),
                                               _lib.stream_ptr(w_raw.device)))


def _wow_scale_fused(lib, src, dst_c, out_w, s, scaling_function, sig_mode, sigma, sigma_e, nz, weight):
    """One fused WOW scale (wb_wow_scale).  Returns False without launching anything when the problem is outside the
    fused kernel (the caller then takes the two-pass route)."""
    b, h, w, pitch, bstride = _frame_layout(src)
    _, _, _, c_pitch, c_bstride = _frame_layout(dst_c)
    _, _, _, w_pitch, w_bstride = _frame_layout(out_w)
    with torch.cuda.device(src.device):
        rc = lib.wb_wow_scale(src.data_ptr(), dst_c.data_ptr(), out_w.data_ptr(), b, h, w, pitch, bstride, c_pitch,
                              c_bstride, w_pitch, w_bstride, s, scaling_function.taps_code, _lib.dtype_code(src.dtype),
                              sig_mode, float(sigma), float(sigma_e), nz.host, nz.dev_ptr, float(weight),
                              _lib.stream_ptr(src.device))
    if rc == _lib.WB_ENOT_FUSABLE:
        return False
    _lib.check(rc)
    return True


def _scalar_noise(noise, device):
    """None -> None; number / 0-d array / 1-element tensor -> _Noise with a host or device scalar."""
    if noise is None:
        return None
    if isinstance(noise, torch.Tensor):
        if noise.numel() == 1 and noise.ndim <= 1 and noise.is_cuda and noise.dtype == torch.float64:
            return _Noise(dev=noise)
        if noise.numel() == 1:
            return _Noise(host=float(noise.item()))
        return "map"
    if isinstance(noise, np.ndarray) and noise.ndim > 0:
        return "map"
    return _Noise(host=float(noise))


_STACK_NOISE_FORMS = "None, a scalar, per-frame scalars (B,), one map (H, W) for every frame or one map per frame (B, H, W)"


def _stack_noise(noise, b, h, w, dtype, device):
    """The ``noise`` of wow_batch / wow_stream for ``b`` frames of (h, w): None, a _Noise with a host or device scalar,
    with float64 per-frame scalars (``dev``, shape (b,)), or with a map (``map``, (h, w) or (b, h, w), frame dtype)."""
    nz = _scalar_noise(noise, device)
    if not isinstance(nz, str):
        return nz
    shape = tuple(noise.shape)
    if shape == (b,):
        t = noise if isinstance(noise, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(noise))
        return _Noise(dev=t.to(device=device, dtype=torch.float64).contiguous())
    if shape in ((h, w), (b, h, w)):
        return _Noise(map_=broadcast_noise_map(noise, shape, dtype, device))
    raise ValueError(f"noise of shape {shape} for {b} frames of {h} x {w}: expected {_STACK_NOISE_FORMS}")


def _blend_options(preserve_variance, gamma, gamma_min, gamma_max, h):
    """The gamma blend (h > 0) and preserve_variance options of wow() for _wow_stack, or None when neither is asked for.
    ``1 / gamma`` is evaluated here when the blend needs it, so that gamma == 0 raises ZeroDivisionError as the
    reference's ``pow(1 / gamma)`` does."""
    if h == 0 and not preserve_variance:
        return None
    if h > 0:
        1 / gamma  # noqa: B018
    return bool(preserve_variance), float(gamma), gamma_min, gamma_max, float(h)


def _wow_stack(stack, scaling_function_class, n_scales, wts, dns, sigma_bilateral, bilateral_scaling, whitening,
               soft_threshold, noise, buffers=None, blend=None):
    """The fused WOW pipeline on a stack (B, H, W) of frames.  Returns (recon (B,H,W), planes (B,L+1,H,W), noise).

    ``buffers``: optional dict of preallocated device tensors (planes, scratch, reconstruction, workspace), filled in
    on first use and reused by later calls with the same geometry (``wow_stream`` keeps one per frame in flight, so
    that its steady state allocates nothing large).

    With whitening and at least one scale, the whole pipeline is ONE library call (wb_wow_cascade, or
    wb_wow_cascade_map for a per-pixel noise map; csrc/cascade.cu holds its per-scale policy).  ``blend`` (from
    _blend_options: preserve_variance, gamma, gamma_min, gamma_max, h) takes wb_wow_cascade_blend, one call for every
    noise form, with or without whitening and for any scale count.  Without whitening and blend, K1/K2 write every
    plane and wb_denoise_plane thresholds and weights it in place, with the MAD noise estimated from plane 0 where a
    threshold first needs it.  Then the residual plane is rescaled (whitening) or weighted and K5 sums the planes.
    The noise is estimated on the device: no host synchronisation anywhere."""
    lib = _lib.load(require_cuda=True)
    sf = scaling_function_class(2)
    b, h, w = stack.shape
    dev, dt = stack.device, stack.dtype
    L = n_scales
    if buffers is None:
        buffers = {}

    def buffer(name, shape):
        t = buffers.get(name)
        if t is None or tuple(t.shape) != tuple(shape) or t.dtype != dt or t.device != dev:
            t = buffers[name] = torch.empty(shape, dtype=dt, device=dev)
        return t

    planes = buffer("planes", (b, L + 1, h, w))
    bilateral = sigma_bilateral
    sigma_e = sf.sigma_e(bilateral=bilateral)
    transform = AtrousTransform(scaling_function_class, bilateral=bilateral, bilateral_scaling=bilateral_scaling)
    factors = transform.var_factors(L) if bilateral is not None else [None] * L
    if blend is not None or (whitening and L >= 1):
        import ctypes
        scratch3 = buffer("scratch3", (3, b, h, w)) if L >= 1 else None
        recon = buffer("recon", (b, h, w))
        code = _lib.dtype_code(dt)
        ws_bytes = (lib.wb_wow_cascade_workspace_bytes if blend is None else
                    lib.wb_wow_cascade_blend_workspace_bytes)(code, b, h * w)
        ws = buffers.get("cascade_ws")
        if ws is None or ws.numel() < ws_bytes or ws.device != dev:
            ws = buffers["cascade_ws"] = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        any_sig = any(d != 0 for d in dns[:L])
        nz_map = None if noise is None else noise.map
        estimate = noise is None and any_sig
        nz = noise
        if estimate:
            nz = _Noise(dev=torch.empty(b, dtype=torch.float64, device=dev))
        use = nz if nz is not None else _Noise()
        arr = ctypes.c_double * (L + 1)
        _, _, _, pitch, bstride = _frame_layout(stack)
        head = (stack.data_ptr(), pitch, bstride, planes.data_ptr(), None if scratch3 is None else scratch3.data_ptr(),
                recon.data_ptr())
        tail = (b, h, w, L, sf.taps_code, code, arr(*[float(x) for x in wts[:L + 1]]),
                arr(*([float(x) for x in dns[:L]] + [0.0])), arr(*([float(x) for x in sigma_e[:L]] + [0.0])),
                None if bilateral is None else arr(*([float(x) for x in factors[:L]] + [0.0])),
                1 if soft_threshold else 0)
        m_pitch = m_bstride = 0
        if nz_map is not None:
            _, _, _, m_pitch, m_bstride = _frame_layout(nz_map)
        with torch.cuda.device(dev):
            if blend is not None:
                pv, gamma, gamma_min, gamma_max, hh = blend
                g = buffer("gamma", (b, h, w)) if hh > 0 else None
                _lib.check(lib.wb_wow_cascade_blend(
                    *head, None if g is None else g.data_ptr(), *tail, float(use.host), use.dev_ptr,
                    1 if estimate else 0, 0 if nz_map is None else 1, None if nz_map is None else nz_map.data_ptr(),
                    m_pitch, m_bstride, 1 if whitening and hh < 1 else 0, 1 if pv else 0, hh, gamma,
                    0.0 if gamma_min is None else float(gamma_min), 0 if gamma_min is None else 1,
                    0.0 if gamma_max is None else float(gamma_max), 0 if gamma_max is None else 1, ws.data_ptr(),
                    ws.numel(), _lib.stream_ptr(dev)))
            elif nz_map is not None:
                _lib.check(lib.wb_wow_cascade_map(*head, *tail, nz_map.data_ptr(), m_pitch, m_bstride, ws.data_ptr(),
                                                  ws.numel(), _lib.stream_ptr(dev)))
            else:
                _lib.check(lib.wb_wow_cascade(*head, *tail, float(use.host), use.dev_ptr, 1 if estimate else 0,
                                              ws.data_ptr(), ws.numel(), _lib.stream_ptr(dev)))
        return recon, planes, nz
    if L == 0:
        planes[:, 0].copy_(stack)
    scratch = buffer("scratch", (2, b, h, w)) if L > 1 else None
    nz = noise  # _Noise or None
    nz_map = None if noise is None else noise.map
    src = stack
    for s in range(L):
        dst_c = planes[:, L] if s == L - 1 else scratch[s & 1]
        d, wt = dns[s], wts[s]
        need_sig = d != 0
        mode = (1 if soft_threshold else 2) if need_sig else 0
        atrous_scale(src, s, sf, out_c=dst_c, out_w=planes[:, s], var_factor=factors[s])
        if need_sig and nz is None:
            nz = _Noise(dev=abs_median_noise(planes[:, 0], sigma_e[0]))
        if mode or wt != 1:
            use = nz if need_sig else _Noise()
            # wb_denoise_plane reads one map plane for every frame: one launch per frame for per-frame maps
            per_frame = need_sig and nz_map is not None and nz_map.ndim == 3
            for f0, nf in ([(f, 1) for f in range(b)] if per_frame else [(0, b)]):
                m_ptr = 0 if not need_sig or nz_map is None else nz_map[f0].data_ptr() if per_frame else \
                    nz_map.data_ptr()
                with torch.cuda.device(dev):
                    _lib.check(lib.wb_denoise_plane(planes[f0, s].data_ptr(), h * w, nf, (L + 1) * h * w,
                                                    _lib.dtype_code(dt), mode, float(d),
                                                    float(sigma_e[s]) if need_sig else 1.0, use.host, use.dev_ptr,
                                                    m_ptr, float(wt), _lib.stream_ptr(dev)))
        src = dst_c
    # residual plane: c_L *= wt_L / std(c_L)  (watroo/utils.py:185-189, :203); with whitening only for L == 0 here
    last = planes[:, L]
    if whitening:
        # (a fused rescale + synthesis pass measured slower: the separate rescale finds c_L still in L2)
        mom = plane_moments(last)
        with torch.cuda.device(dev):
            _lib.check(lib.wb_residual_rescale(last.data_ptr(), h * w, b, (L + 1) * h * w, _lib.dtype_code(dt),
                                               mom.data_ptr(), float(wts[L]), _lib.stream_ptr(dev)))
    elif wts[L] != 1:
        last.mul_(wts[L])
    recon = synthesis(planes, out=buffer("recon", (b, h, w)))
    return recon, planes, nz


def wow(data, scaling_function=B3spline, n_scales=None, weights=[], whitening=True, denoise_coefficients=[],
        noise=None, bilateral=None, bilateral_scaling=False, soft_threshold=True, preserve_variance=False, gamma=3.2,
        gamma_min=None, gamma_max=None, h=0):
    """Wavelets Optimized Whitening (watroo/utils.py:105-219): ``(recon, coefficients)``.

    ``data`` is a 2-D image (ndarray or torch tensor) or a ``Coefficients`` object (which is then whitened in
    place, as in the reference).  For an image every option runs as one library call: the ``bilateral`` /
    ``denoise_coefficients`` / ``weights`` / ``whitening`` / ``noise`` options on the fused kernels, and ``h > 0`` (gamma
    blending, utils.py:157-158, :207-217) and ``preserve_variance`` (utils.py:178-184) on wb_wow_cascade_blend.
    ``Coefficients`` input with those two options takes a plane-by-plane route over the same kernels."""
    general = h != 0 or preserve_variance
    if isinstance(data, Coefficients):
        if general:
            return _wow_general(data, weights, whitening, denoise_coefficients, bilateral, soft_threshold,
                                preserve_variance, gamma, gamma_min, gamma_max, h)
        return _wow_coefficients(data, weights, whitening, denoise_coefficients, bilateral, soft_threshold)
    if not isinstance(data, (np.ndarray, torch.Tensor)):
        raise ValueError("Unknown input type")  # watroo/utils.py:133
    img, was_numpy = to_device_image(data, ndim_ok=(1, 2, 3))
    if img.ndim != 2:
        # 1-D signals and 3-D volumes: the reference's loop is dimension-generic (watroo/utils.py:148-150, :194)
        n_scales, sigma_bilateral, wts, dns = _wow_plan(img.shape, scaling_function, n_scales, weights,
                                                        denoise_coefficients, bilateral, h=h, n_dims=img.ndim)
        if img.ndim == 3 and sigma_bilateral is None and h == 0 and not preserve_variance and n_scales >= 0:
            recon, co = _wow_volume(img, scaling_function, n_scales, wts, dns, whitening, soft_threshold, noise)
            return _result(recon, was_numpy), co
        transform = AtrousTransform(scaling_function, bilateral=sigma_bilateral, bilateral_scaling=bilateral_scaling)
        co = transform(img, n_scales)
        co.noise = noise
        recon = _wow_nd(co, wts, dns, whitening, soft_threshold, preserve_variance, gamma, gamma_min, gamma_max, h)
        return _result(recon, was_numpy), co
    n_scales, sigma_bilateral, wts, dns = _wow_plan(img.shape, scaling_function, n_scales, weights,
                                                    denoise_coefficients, bilateral, h=h)
    blend = _blend_options(preserve_variance, gamma, gamma_min, gamma_max, h)
    nz = _scalar_noise(noise, img.device)
    if isinstance(nz, str):
        # a per-pixel noise map, broadcast to the image: two passes at every scale, the map applied inside K3
        nz = _Noise(map_=broadcast_noise_map(noise, img.shape, img.dtype, img.device))
    recon, planes, nz = _wow_stack(img.unsqueeze(0), scaling_function, n_scales, wts, dns, sigma_bilateral,
                                   bilateral_scaling, whitening, soft_threshold, nz, blend=blend)
    co = Coefficients(planes[0], scaling_function(2), sigma_bilateral)
    if blend is not None and noise is not None:
        # the noise as Coefficients._noise_arg leaves it: an array map that a threshold used is kept as its device copy
        used = isinstance(noise, np.ndarray) and noise.ndim > 0 and any(d != 0 for d in dns[:n_scales])
        co.noise = nz.map if used else noise
    elif nz is not None and nz.map is not None:
        co.noise = noise
    elif nz is not None:
        co.noise = nz.dev if nz.dev is not None else nz.host
    else:
        co.noise = None
    return _result(recon[0], was_numpy), co


def _volume_noise(noise, shape, dtype, device, thresholded):
    """The noise of wow() on a volume of ``shape`` (D, H, W), classified as Coefficients._noise_arg classifies it.
    Returns (_Noise or None for the MAD estimate, map z-stride, the noise the coefficients keep afterwards)."""
    d, h, w = shape
    if noise is None:
        return None, 0, None
    if isinstance(noise, torch.Tensor) and not (noise.numel() == 1 and noise.ndim <= 1):
        m, kept = noise, noise
    elif isinstance(noise, np.ndarray) and noise.ndim > 0:
        m, kept = noise, None  # a map that a threshold uses is kept as its device copy
    else:
        if isinstance(noise, torch.Tensor):
            nz = _Noise(dev=noise) if noise.is_cuda and noise.dtype == torch.float64 else _Noise(host=float(noise.item()))
        elif isinstance(noise, np.ndarray) or isinstance(noise, numbers.Number):
            nz = _Noise(host=float(noise))
        elif thresholded:
            raise TypeError(f"unsupported noise type {type(noise)}")
        else:
            nz = _Noise()
        return nz, 0, noise
    if not thresholded:
        return _Noise(), 0, noise
    if tuple(m.shape) in ((h, w), (1, h, w)):
        # one (H, W) map for every slice: read with a depth stride of 0
        plane = broadcast_noise_map(m.reshape(h, w), (h, w), dtype, device)
        return _Noise(map_=plane), 0, kept if kept is not None else plane.expand(d, h, w)
    full = broadcast_noise_map(m, shape, dtype, device)
    return _Noise(map_=full), h * w, kept if kept is not None else full


def _wow_volume(img, scaling_function, n_scales, wts, dns, whitening, soft_threshold, noise):
    """wow() of a plain volume (D, H, W) with h == 0 and no preserve_variance: one wb_wow_cascade_volume call,
    bit-identical to the transform followed by _wow_nd, the noise left on the coefficients as _wow_nd leaves it."""
    lib = _lib.load(require_cuda=True)
    sf = scaling_function(3)
    img = img.contiguous()
    dev, dt = img.device, img.dtype
    code = _lib.dtype_code(dt)
    L = n_scales
    shape = tuple(img.shape)
    planes = torch.empty((L + 1,) + shape, dtype=dt, device=dev)
    recon = torch.empty(shape, dtype=dt, device=dev)
    scratch = torch.empty(lib.wb_volume_scratch_bytes(code, *shape, L), dtype=torch.uint8, device=dev)
    ws = torch.empty(lib.wb_wow_cascade_volume_workspace_bytes(code, *shape), dtype=torch.uint8, device=dev)
    thresholded = any(d != 0 for d in dns[:L])
    nz, zstride, kept = _volume_noise(noise, shape, dt, dev, thresholded)
    estimate = nz is None and thresholded
    if estimate:
        nz = _Noise(dev=torch.empty(1, dtype=torch.float64, device=dev))
        kept = nz.dev
    use = nz if nz is not None else _Noise()
    sigma_e = sf.sigma_e()
    arr = ctypes.c_double * (L + 1)
    with torch.cuda.device(dev):
        _lib.check(lib.wb_wow_cascade_volume(
            img.data_ptr(), planes.data_ptr(), scratch.data_ptr(), recon.data_ptr(), *shape, L, sf.taps_code, code,
            arr(*[float(x) for x in wts[:L + 1]]), arr(*([float(x) for x in dns[:L]] + [0.0])),
            arr(*([float(x) for x in sigma_e[:L]] + [0.0])), 1 if soft_threshold else 0, 1 if whitening else 0,
            float(use.host), use.dev_ptr, 1 if estimate else 0, use.map_ptr or None, zstride, ws.data_ptr(), ws.numel(),
            _lib.stream_ptr(dev)))
    co = Coefficients(planes, sf, None)
    co.noise = kept
    return recon, co


def _wow_nd(co, wts, dns, whitening, soft_threshold, preserve_variance, gamma, gamma_min, gamma_max, h, smooth=None):
    """The loop of wow() (watroo/utils.py:172-217) on the coefficients of a 1-D signal or a 3-D volume, every option
    included: the transform and the n-D smooth of the local power run in the library's kernels, the plane-wise factors
    are element-wise device arithmetic in the reference's order and dtypes.  A parity path, whitened in place.
    ``smooth``: the n-D smooth of the local power (default _smooth_nd)."""
    from .wavelets import _smooth_nd
    smooth = smooth or _smooth_nd
    data = co.data
    dt = data.dtype
    L = len(co) - 1
    white = whitening and h < 1
    gamma_scaled = torch.zeros_like(data[0]) if h > 0 else None
    for s in range(L + 1):
        c = data[s]
        power = c * c
        power_norm = None
        if preserve_variance:  # utils.py:178-184
            power_norm = c.to(torch.float64).std(unbiased=False).to(dt) if s == L else torch.sqrt(power.mean())
        if s == L:
            local_power = None
            if white:
                sd = plane_moments(c.reshape(1, -1))[0, 2].to(dt)
                local_power = torch.where(sd <= 0, torch.full_like(sd, 1e-15), sd)
        else:
            local_power = None
            if white:
                local_power = smooth(power.contiguous(), s, co.scaling_function)  # plain smooth, utils.py:194
                local_power = torch.sqrt(torch.where(local_power <= 0, torch.full_like(local_power, 1e-15), local_power))
            sig = co.significance(dns[s], s, soft_threshold=soft_threshold)
            if sig.dtype == torch.bool or sig.dtype == torch.float64:
                c.copy_((c.to(torch.float64) * sig.to(torch.float64)).to(dt))  # product in float64, rounded once
        if gamma_scaled is not None:
            gamma_scaled += c
        factor = torch.as_tensor(wts[s], dtype=dt, device=c.device)
        if power_norm is not None:
            factor = factor * power_norm
        if local_power is not None:
            factor = factor / local_power
        c.mul_(factor)
    recon = synthesis(data.reshape(L + 1, 1, -1)).reshape(data.shape[1:])
    if gamma_scaled is not None:  # utils.py:207-217
        lo = gamma_scaled.min() if gamma_min is None else gamma_min
        hi = gamma_scaled.max() if gamma_max is None else gamma_max
        gamma_scaled -= lo
        gamma_scaled /= (hi - lo)
        gamma_scaled.clamp_(0, 1)
        gamma_scaled.pow_(1 / gamma)
        recon = (1 - h) * recon + h * gamma_scaled
    return recon


def wow_batch(frames, scaling_function=B3spline, n_scales=None, weights=[], whitening=True, denoise_coefficients=[],
              noise=None, bilateral=None, bilateral_scaling=False, soft_threshold=True, preserve_variance=False,
              gamma=3.2, gamma_min=None, gamma_max=None, h=0):
    """NEW entry point (no reference equivalent): WOW of a stack ``(B, H, W)`` of independent frames, every kernel
    launched once for the whole stack.  Returns ``(recon (B,H,W), planes (B,L+1,H,W), noise)`` as device tensors;
    per-frame results are identical to ``wow(frame, noise=<that frame's noise>, ...)``.

    ``noise`` (NumPy or torch): None (MAD estimate per frame), a scalar, per-frame scalars ``(B,)``, one per-pixel map
    ``(H, W)`` for every frame or one map per frame ``(B, H, W)``; anything else raises ValueError.  The returned noise
    is the one used: the (B,) float64 estimates or scalars, the scalar, or the map in the frame dtype.

    ``h > 0`` blends every frame with its own gamma-stretched image; ``gamma_min`` / ``gamma_max`` of None take that
    frame's min / max, as ``wow`` does frame by frame."""
    stack, _ = to_device_image(frames, ndim_ok=(3,))
    n_scales, sigma_bilateral, wts, dns = _wow_plan(stack.shape[1:], scaling_function, n_scales, weights,
                                                    denoise_coefficients, bilateral, h=h)
    blend = _blend_options(preserve_variance, gamma, gamma_min, gamma_max, h)
    b, fh, fw = stack.shape
    nz = _stack_noise(noise, b, fh, fw, stack.dtype, stack.device)
    recon, planes, nz = _wow_stack(stack, scaling_function, n_scales, wts, dns, sigma_bilateral, bilateral_scaling,
                                   whitening, soft_threshold, nz, blend=blend)
    if nz is None:
        noise_out = None
    elif nz.map is not None:
        noise_out = nz.map
    else:
        noise_out = nz.dev if nz.dev is not None else nz.host
    return recon, planes, noise_out


def wow_stream(frames, out=None, depth=2, scaling_function=B3spline, **kwargs):
    """NEW entry point (no reference equivalent): ``wow()`` of a sequence of HOST frames ``(N, H, W)`` into a host array
    ``(N, H, W)`` of reconstructions, overlapping the host->device copy of frame n+1, the WOW of frame n and the
    device->host copy of the reconstruction of frame n-1 on three CUDA streams (``depth`` device buffers in flight).

    ``frames`` / ``out``: torch CPU tensors (pinned memory is used as is, pageable memory is staged through a pinned copy)
    or NumPy arrays; ``kwargs`` are those of ``wow``.  ``noise`` takes the forms of ``wow_batch`` with N frames: a
    scalar, per-frame scalars ``(N,)`` and one map ``(H, W)`` are uploaded once; host maps ``(N, H, W)`` are streamed
    next to their frames (one device map buffer per frame in flight).  Returns ``out`` (allocated pinned when None; a
    NumPy view of it for NumPy input).  Per-frame results are identical to ``wow(frame, noise=<its noise>, ...)[0]``."""
    was_numpy = not isinstance(frames, torch.Tensor)
    host = torch.from_numpy(np.ascontiguousarray(frames)) if was_numpy else frames
    if host.ndim != 3:
        raise ValueError("wow_stream() takes a stack of frames (N, H, W)")
    if host.is_cuda:
        raise ValueError("wow_stream() takes host frames; use wow_batch() for device-resident stacks")
    if host.dtype not in (torch.float32, torch.float64):
        host = host.to(torch.float64)  # the reference's recast rule for integer inputs
    if not host.is_pinned():
        host = host.contiguous().pin_memory()
    n, h, w = host.shape
    if out is None:
        out = torch.empty((n, h, w), dtype=host.dtype).pin_memory()
    out_t = torch.from_numpy(out) if isinstance(out, np.ndarray) else out
    if tuple(out_t.shape) != (n, h, w) or out_t.dtype != host.dtype:
        raise ValueError("out must be (N, H, W) of the frame dtype")
    staged = None if out_t.is_pinned() else torch.empty(out_t.shape, dtype=out_t.dtype).pin_memory()
    dst = out_t if staged is None else staged
    _lib.load(require_cuda=True)
    dev = torch.device("cuda", torch.cuda.current_device())
    depth = max(1, min(int(depth), n))
    s_in, s_cmp, s_out = _pipeline_streams(dev)
    caller = torch.cuda.current_stream(dev)
    for st in (s_in, s_cmp, s_out):
        st.wait_stream(caller)
    # Every option is planned ONCE and every frame in flight owns one set of device buffers (planes, scratch, gamma
    # plane, reconstruction): after the first `depth` frames nothing large is allocated -- with wow() called per frame
    # the caching allocator split and re-grew its blocks while the host ran ahead of the device (a cudaMalloc of 0.7 GB
    # per frame: 25 ms instead of 1.3).
    opts = dict(kwargs)
    unknown = set(opts) - {"n_scales", "weights", "whitening", "denoise_coefficients", "noise", "bilateral",
                           "bilateral_scaling", "soft_threshold", "preserve_variance", "gamma", "gamma_min", "gamma_max", "h"}
    if unknown:
        raise TypeError(f"wow_stream() got unexpected keyword arguments {sorted(unknown)}")
    noise = opts.get("noise")
    # per-frame noise: a device vector of scalars (sliced per frame), or the (N, H, W) maps streamed with the frames
    nz_vec = map_host = None
    nz0 = None
    if noise is not None and tuple(getattr(noise, "shape", ())) == (n, h, w) and not getattr(noise, "is_cuda", False):
        map_host = torch.from_numpy(np.ascontiguousarray(noise)) if not isinstance(noise, torch.Tensor) else noise
        map_host = map_host.to(host.dtype)
        if not map_host.is_pinned():
            map_host = map_host.contiguous().pin_memory()
    else:
        nz0 = _stack_noise(noise, n, h, w, host.dtype, dev)
        if nz0 is not None and ((nz0.dev is not None and nz0.dev.numel() > 1) or
                                (nz0.map is not None and nz0.map.ndim == 3)):
            nz_vec, nz0 = nz0, None
        s_cmp.wait_stream(caller)  # the noise was uploaded on the caller's stream
    blend_h = opts.get("h", 0)
    L, sigma_bilateral, wts, dns = _wow_plan((h, w), scaling_function, opts.get("n_scales"), opts.get("weights", []),
                                             opts.get("denoise_coefficients", []), opts.get("bilateral"), h=blend_h)
    blend = _blend_options(opts.get("preserve_variance", False), opts.get("gamma", 3.2), opts.get("gamma_min"),
                           opts.get("gamma_max"), blend_h)
    bil_scaling, whitening, soft = (opts.get("bilateral_scaling", False), opts.get("whitening", True),
                                    opts.get("soft_threshold", True))
    d_in = [torch.empty((h, w), dtype=host.dtype, device=dev) for _ in range(depth)]
    d_map = [torch.empty((h, w), dtype=host.dtype, device=dev) for _ in range(depth)] if map_host is not None else None
    d_out = [None] * depth
    bufs = [dict() for _ in range(depth)]
    ev_in = [torch.cuda.Event() for _ in range(depth)]
    ev_cmp = [torch.cuda.Event() for _ in range(depth)]
    ev_out = [torch.cuda.Event() for _ in range(depth)]
    for i in range(n):
        b = i % depth
        with torch.cuda.stream(s_in):
            if i >= depth:
                s_in.wait_event(ev_cmp[b])       # the WOW that read d_in[b] is done
            d_in[b].copy_(host[i], non_blocking=True)
            if d_map is not None:
                d_map[b].copy_(map_host[i], non_blocking=True)
            ev_in[b].record(s_in)
        with torch.cuda.stream(s_cmp):
            s_cmp.wait_event(ev_in[b])
            if i >= depth:
                s_cmp.wait_event(ev_out[b])      # the download of d_out[b] is done (its memory is reused)
            if d_map is not None:
                nz_i = _Noise(map_=d_map[b])
            elif nz_vec is not None:
                nz_i = _Noise(dev=nz_vec.dev[i:i + 1]) if nz_vec.dev is not None else _Noise(map_=nz_vec.map[i])
            else:
                nz_i = nz0
            recon, _, _ = _wow_stack(d_in[b].unsqueeze(0), scaling_function, L, wts, dns, sigma_bilateral, bil_scaling,
                                     whitening, soft, nz_i, buffers=bufs[b], blend=blend)
            d_out[b] = recon[0]
            ev_cmp[b].record(s_cmp)
        with torch.cuda.stream(s_out):
            s_out.wait_event(ev_cmp[b])
            dst[i].copy_(d_out[b], non_blocking=True)
            ev_out[b].record(s_out)
    for st in (s_in, s_cmp, s_out):
        caller.wait_stream(st)
    s_out.synchronize()  # the result lives in host memory: hand it back complete
    if staged is not None:
        out_t.copy_(staged)
    return out if (isinstance(out, np.ndarray) or not was_numpy) else out_t.numpy()


def _wow_coefficients(co, weights, whitening, denoise_coefficients, bilateral, soft_threshold, plan=None):
    """wow() on already computed coefficients (watroo/utils.py:128-131, :152-153): planes are whitened in place,
    in plane order, with the lazily estimated noise of the object."""
    lib = _lib.load(require_cuda=True)
    sf = co.scaling_function
    if plan is None:
        n_scales, _, wts, dns = _wow_plan(co.data.shape[1:], sf.__class__, None, weights, denoise_coefficients,
                                          bilateral, from_coefficients=co)
        if n_scales != len(co) - 1:
            n_scales = len(co) - 1  # the warning branch cannot add planes to existing coefficients
    else:
        n_scales, _, wts, dns = plan
    data = co.data
    L = n_scales
    tmp = torch.empty_like(data[0])
    for s in range(L):
        d, wt = dns[s], wts[s]
        plane = data[s]
        if whitening:
            # local power from the raw plane, significance from the raw plane, then both factors (utils.py:194-203)
            nz = co._noise_arg(d) if d != 0 else _Noise()
            if nz.map is not None:
                _whiten_scale_map(lib, plane, tmp, nz.map, s, sf, soft_threshold, d, co.sigma_e[s], wt)
            else:
                mode = (1 if soft_threshold else 2) if d != 0 else 0
                _whiten_scale(lib, plane, tmp, s, sf, mode, d, co.sigma_e[s] if d != 0 else 1.0, nz, wt)
            plane.copy_(tmp)
        else:
            co._denoise_plane(lib, s, d, wt, soft_threshold)
    last = data[L]
    if whitening:
        mom = plane_moments(last)
        with torch.cuda.device(last.device):
            _lib.check(lib.wb_residual_rescale(last.data_ptr(), last.numel(), 1, 0, _lib.dtype_code(last.dtype),
                                               mom.data_ptr(), float(wts[L]), _lib.stream_ptr(last.device)))
    elif wts[L] != 1:
        last.mul_(wts[L])
    return synthesis(data), co


def _wow_general(co, weights, whitening, denoise_coefficients, bilateral, soft_threshold, preserve_variance, gamma,
                 gamma_min, gamma_max, h, plan=None):
    """wow() with the gamma blend (h > 0) and / or preserve_variance (watroo/utils.py:157-158, :174-217), plane by
    plane on raw coefficients: the same kernels as the fused route (K3 whitening, significance, moments, synthesis)
    plus a few device-scalar multiplications; nothing synchronises with the host."""
    lib = _lib.load(require_cuda=True)
    sf = co.scaling_function
    if plan is None:
        n_scales, _, wts, dns = _wow_plan(co.data.shape[1:], sf.__class__, None, weights, denoise_coefficients,
                                          bilateral, from_coefficients=co, h=h)
        n_scales = len(co) - 1
    else:
        n_scales, wts, dns = plan
    data = co.data
    dt = data.dtype
    L = n_scales
    white = whitening and h < 1  # utils.py:186, :193
    gamma_scaled = torch.zeros_like(data[0]) if h > 0 else None
    tmp = torch.empty_like(data[0]) if white else None
    for s in range(L):
        d, wt = dns[s], wts[s]
        plane = data[s]
        power_norm = None
        if preserve_variance:
            mom = plane_moments(plane)[0]                       # [mean, var, std] of the raw plane, float64
            power_norm = torch.sqrt(mom[1] + mom[0] * mom[0]).to(dt)  # sqrt(mean(c**2)), utils.py:182
        nz = co._noise_arg(d) if d != 0 else _Noise()           # lazily, from the current plane 0 (wavelets.py:131)
        if white:
            if nz.map is not None:
                _whiten_scale_map(lib, plane, tmp, nz.map, s, sf, soft_threshold, d, co.sigma_e[s], wt)
            else:
                mode = (1 if soft_threshold else 2) if d != 0 else 0
                _whiten_scale(lib, plane, tmp, s, sf, mode, d, co.sigma_e[s] if d != 0 else 1.0, nz, wt)
        co._denoise_plane(lib, s, d, 1, soft_threshold)         # plane <- raw * significance
        if gamma_scaled is not None:
            gamma_scaled += plane                               # utils.py:200-201: after significance, before weighting
        if white:
            plane.copy_(tmp if power_norm is None else tmp * power_norm)
        else:
            factor = wt if power_norm is None else power_norm * wt
            if power_norm is not None or wt != 1:
                plane.mul_(factor)
    last = data[L]
    mom = plane_moments(last)[0] if (preserve_variance or white) else None
    if gamma_scaled is not None:
        gamma_scaled += last
    factor = torch.ones((), dtype=torch.float64, device=last.device) * wts[L]
    if preserve_variance:
        factor = factor * mom[2].to(dt).to(torch.float64)       # power_norm = np.std(c), utils.py:180
    if white:
        std = mom[2].to(dt).to(torch.float64)
        factor = factor / torch.where(std <= 0, torch.full_like(std, 1e-15), std)  # utils.py:187-189
    last.mul_(factor.to(dt))
    recon = synthesis(data)
    if gamma_scaled is not None:  # utils.py:207-217
        lo = gamma_scaled.min() if gamma_min is None else gamma_min
        hi = gamma_scaled.max() if gamma_max is None else gamma_max
        gamma_scaled -= lo
        gamma_scaled /= (hi - lo)
        gamma_scaled.clamp_(0, 1)
        gamma_scaled.pow_(1 / gamma)
        recon = (1 - h) * recon + h * gamma_scaled
    return recon, co


# ---------------------------------------------------------------------------------------------------------------
# Callers of the transform beyond denoise / wow (SURVEY.md 8(f) ranks 3-4): enhance, richardson_lucy
# ---------------------------------------------------------------------------------------------------------------
def prepare_params(param, ndims):
    """Per-channel parameter lists of ``enhance`` (watroo/utils.py:10-33), quirks included (a scalar given for a
    3-channel image becomes the SAME inner list for every channel)."""
    if ndims == 2:
        if param is None:
            return []
        if type(param) is not list:
            return [param]
        return copy.copy(param)
    if type(param) is not list:
        return [[], ] * ndims if param is None else [[param], ] * ndims
    if len(param) != ndims:
        raise ValueError("Invalid number of parameters")
    out = [prepare_params(p, 2) for p in param]
    if None in out:
        out[out.index(None)] = []
    return out


def enhance(*args, weights=None, denoise=None, soft_threshold=True, out=None, **kwargs):
    """De-noising and / or enhancement by modification of the wavelet coefficients (watroo/utils.py:36-80): per
    channel (a 3-D input is three channels, channel first) transform -> ``Coefficients.denoise(denoise,
    weights=weights)`` -> sum of the planes.  ``args[1]``, when given, is the noise (per channel for 3 channels);
    ``kwargs`` go to ``AtrousTransform``.  NumPy in -> NumPy out (``out`` is filled when given)."""
    img = args[0]
    was_numpy = not isinstance(img, torch.Tensor)
    ndim = img.ndim
    channels = [0, 1, 2] if ndim == 3 else [Ellipsis]
    weights = prepare_params(weights, ndim)
    denoise_p = prepare_params(denoise, ndim)
    atrous = AtrousTransform(**kwargs)
    results = []
    for c in channels:
        dns = denoise_p if c is Ellipsis else denoise_p[c]
        wgt = weights if c is Ellipsis else weights[c]
        if len(wgt) < len(dns):
            wgt.extend([1] * (len(dns) - len(wgt)))
        elif len(dns) < len(wgt):
            dns.extend([0] * (len(wgt) - len(dns)))
        coeffs = atrous(img[c], len(wgt))
        if len(args) == 2:
            coeffs.noise = args[1] if c is Ellipsis else args[1][c]
        else:
            coeffs.noise = coeffs.get_noise()
        coeffs.denoise(dns, weights=wgt, soft_threshold=soft_threshold)
        results.append(synthesis(coeffs.data))
    res = results[0] if ndim != 3 else torch.stack(results)
    if out is not None:
        if isinstance(out, torch.Tensor):
            out.copy_(res)
        else:
            out[...] = res.cpu().numpy()
        return out
    return _result(res, was_numpy)


def _filter2d(img, kernel_dev, flip):
    """cv2.filter2D(img, -1, kernel, (-1,-1), 0, BORDER_REFLECT) on the device (wb_filter2d); flip rotates the kernel."""
    lib = _lib.load(require_cuda=True)
    out = torch.empty_like(img)
    kh, kw = kernel_dev.shape
    with torch.cuda.device(img.device):
        _lib.check(lib.wb_filter2d(img.data_ptr(), out.data_ptr(), img.shape[0], img.shape[1], img.stride(0),
                                   out.stride(0), kernel_dev.data_ptr(), kh, kw, 1 if flip else 0,
                                   _lib.dtype_code(img.dtype), _lib.stream_ptr(img.device)))
    return out


def richardson_lucy(data, psf, iterations=10, denoise_coefficients=(5, 2, 1), threshold_type='soft',
                    uniform_init=False, persistent_mrs=True, fft=False):
    """Wavelet-regularised Richardson-Lucy deconvolution (watroo/utils.py:222-290), every step on the device.

    Per iteration: phi = psf (*) psi (cv2.filter2D with the flipped PSF and the symmetric border, or a circular FFT
    convolution when ``fft``), residual ``data - phi`` -> à trous transform -> significance of every scale against the
    noise of the FIRST transform -> multiresolution support (persistent or not; hard: a mask that only grows, soft: a
    running product applied with the exponent 1/(iteration+1)) -> synthesis -> ``(res + phi) / phi`` -> correlation
    with the PSF -> multiplicative update of psi.  Returns psi (NumPy for NumPy input)."""
    img, was_numpy = to_device_image(data)
    soft = threshold_type == 'soft'
    level = len(denoise_coefficients)
    psf_t = torch.as_tensor(np.ascontiguousarray(psf) if not isinstance(psf, torch.Tensor) else psf)
    psf_dev = psf_t.to(device=img.device, dtype=img.dtype).contiguous()
    transform = AtrousTransform()
    coefficients = transform(img, level)
    if uniform_init:
        psi = torch.ones(img.shape, dtype=torch.float32, device=img.device)
        psi *= (img.sum() / img.numel()).to(torch.float32)
    else:
        coefficients.denoise(denoise_coefficients, soft_threshold=soft)
        psi = synthesis(coefficients.data)
    mrs = (torch.ones if soft else torch.zeros)((level,) + tuple(img.shape), dtype=torch.float64, device=img.device)
    if fft:
        h, w = psi.shape
        kh, kw = psf_dev.shape
        padded = torch.zeros_like(psi)
        padded[h // 2 - kh // 2: h // 2 - kh // 2 + kh, w // 2 - kw // 2: w // 2 - kw // 2 + kw] = psf_dev
        # np.fft computes in float64 whatever the input dtype: the reference's fft route runs in double from here on
        fft_psf = torch.fft.rfft2(torch.roll(padded, (h // 2, w // 2), dims=(0, 1)).to(torch.float64))
        psf_conj = fft_psf.conj()
    for iteration in range(iterations):
        if fft:
            phi = torch.fft.irfft2(torch.fft.rfft2(psi.to(torch.float64)) * fft_psf, s=psi.shape)
        else:
            phi = _filter2d(psi.to(img.dtype) if psi.dtype != img.dtype else psi, psf_dev, flip=True)
        res = img - phi
        res_coefficients = transform(res, level)
        res_coefficients._noise = coefficients._noise  # None when uniform_init: then estimated from the residual
        for s, c in enumerate(denoise_coefficients):
            sig = res_coefficients.significance(c, s, soft_threshold=soft)
            plane = res_coefficients.data[s]
            if not soft:
                sig = sig.to(torch.bool) if sig.dtype != torch.bool else sig
                if persistent_mrs:
                    mrs[s][sig] = 1
                else:
                    mrs[s] = sig.to(torch.float64)
                plane.copy_((plane.to(torch.float64) * mrs[s]).to(plane.dtype))
            else:
                if persistent_mrs:
                    mrs[s] *= sig.to(torch.float64)
                else:
                    mrs[s] = sig.to(torch.float64)
                plane.copy_((plane.to(torch.float64) * mrs[s] ** (1 / (iteration + 1))).to(plane.dtype))
        res = synthesis(res_coefficients.data)
        res += phi
        res /= phi
        if fft:
            conv = torch.fft.irfft2(torch.fft.rfft2(res.to(torch.float64)) * psf_conj, s=res.shape)
        else:
            conv = _filter2d(res, psf_dev, flip=False)
        psi = psi * conv.to(psi.dtype)
    return _result(psi, was_numpy)
