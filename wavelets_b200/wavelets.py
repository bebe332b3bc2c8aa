"""Host-side mirror of the reference's transform API (watroo/wavelets.py:108-149, :290-444) on top of the C ABI.

``AtrousTransform(Triangle|B3spline)(img, n_scales)`` returns a ``Coefficients`` object whose ``.data`` is a torch
CUDA tensor of shape ``(n_scales + 1, H, W)`` holding ``[w_0 .. w_{L-1}, c_L]``.  Inputs may be NumPy arrays (copied
to the current CUDA device) or torch tensors.  All arithmetic runs in the sm_100a kernels of
``libwavelets_b200.so``; there is no CPU path.
"""
from __future__ import annotations

import copy
import numbers

import numpy as np
import torch

from . import _lib
from .scaling import AbstractScalingFunction, B3spline, Triangle

__all__ = ["AtrousTransform", "B3spline", "Triangle", "Coefficients", "atrous_scale", "convolution"]

# integer / big-endian inputs are recast to float64 (watroo/wavelets.py:297, :319-320)
_RECAST_NUMPY = tuple(np.dtype(t) for t in (np.int16, np.uint16, np.int32, np.uint32, np.int64, ">f4", ">f8"))
_RECAST_TORCH = (torch.int16, torch.int32, torch.int64)


def _device():
    _lib.load(require_cuda=True)
    return torch.device("cuda", torch.cuda.current_device())


def to_device_image(arr, ndim_ok=(2,)):
    """Bring an image to the device as a float32/float64 tensor with unit inner stride.

    Returns (tensor, was_numpy).  Follows the reference's dtype rule: float32/float64 pass through, the integer
    and big-endian types of ``_recasting_types`` become float64; anything else is rejected (the reference silently
    computes in uint8 or crashes inside OpenCV for float16 -- neither is worth reproducing)."""
    was_numpy = not isinstance(arr, torch.Tensor)
    if was_numpy:
        arr = np.asarray(arr)
        if arr.ndim > 3:
            raise ValueError("Unsupported number of dimensions")  # watroo/wavelets.py:316-317
        if arr.dtype in _RECAST_NUMPY:
            arr = arr.astype(np.float64)
        if arr.dtype not in (np.dtype(np.float32), np.dtype(np.float64)):
            raise TypeError(f"unsupported image dtype {arr.dtype}: expected float32/float64 or a recast integer type")
        t = torch.from_numpy(np.ascontiguousarray(arr)).to(_device(), non_blocking=False)
    else:
        if arr.ndim > 3:
            raise ValueError("Unsupported number of dimensions")
        t = arr
        if t.dtype in _RECAST_TORCH:
            t = t.to(torch.float64)
        if t.dtype not in (torch.float32, torch.float64):
            raise TypeError(f"unsupported image dtype {t.dtype}: expected float32/float64 or a recast integer type")
        if not t.is_cuda:
            t = t.to(_device(), non_blocking=True)
        if t.stride(-1) != 1:
            t = t.contiguous()
    if t.ndim not in ndim_ok:
        if t.ndim == 3 or t.ndim == 1:
            raise NotImplementedError(
                "this entry point takes 2-D images; a 3-D input is a volume in the reference "
                "(watroo/wavelets.py:322), not a batch -- use AtrousTransform.batch() / wow_batch() for stacks of frames")
        raise ValueError("Unsupported number of dimensions")
    return t, was_numpy


def _frame_layout(t):
    """(batch, H, W, pitch, bstride) of a 2-D image or a 3-D stack with unit inner stride."""
    if t.ndim == 2:
        return 1, t.shape[0], t.shape[1], t.stride(0), 0
    return t.shape[0], t.shape[1], t.shape[2], t.stride(1), t.stride(0)


def _out_args(t):
    if t is None or t is False:
        return 0, 0, 0
    _, _, _, pitch, bstride = _frame_layout(t)
    return t.data_ptr(), pitch, bstride


def atrous_scale(src, scale, scaling_function, out_c=None, out_w=None, var_factor=None):
    """One scale of the cascade on device tensors: ``out_c = S_scale[src]`` (or its bilateral variant when
    ``var_factor`` is given), ``out_w = src - out_c``.

    Thin wrapper over ``wb_atrous_scale`` / ``wb_atrous_scale_bilateral``.  ``src`` is (H, W) or (B, H, W); outputs
    are allocated when not given (pass ``False`` to skip one)."""
    lib = _lib.load(require_cuda=True)
    b, h, w, pitch, bstride = _frame_layout(src)
    if out_c is None:
        out_c = torch.empty(src.shape, dtype=src.dtype, device=src.device)
    if out_w is None:
        out_w = torch.empty(src.shape, dtype=src.dtype, device=src.device)
    pc, c_pitch, c_bs = _out_args(out_c)
    pw, w_pitch, w_bs = _out_args(out_w)
    with torch.cuda.device(src.device):
        if var_factor is None:
            _lib.check(lib.wb_atrous_scale(src.data_ptr(), pc, pw, b, h, w, pitch, bstride, c_pitch, c_bs, w_pitch,
                                           w_bs, int(scale), scaling_function.taps_code, _lib.dtype_code(src.dtype),
                                           _lib.stream_ptr(src.device)))
        else:
            _lib.check(lib.wb_atrous_scale_bilateral(src.data_ptr(), pc, pw, b, h, w, pitch, bstride, c_pitch, c_bs,
                                                     w_pitch, w_bs, int(scale), scaling_function.taps_code,
                                                     _lib.dtype_code(src.dtype), float(var_factor),
                                                     _lib.stream_ptr(src.device)))
    return (None if out_c is False else out_c), (None if out_w is False else out_w)


def convolution(arr, scaling_function, s=0, output=None):
    """Device counterpart of the reference's exported ``convolution`` (watroo/wavelets.py:35-45): the dilated smooth
    ``S_s[arr]`` with the reference's border (2-D / 3-D: symmetric, 1-D: whole-sample mirror).

    NumPy in -> NumPy out, torch tensor in -> device tensor out.  ``output`` (the reference's in-place argument) may be a
    device tensor (written directly when 2-D) or an ndarray (filled from the device result); it is returned."""
    img, was_numpy = to_device_image(arr, ndim_ok=(1, 2, 3))
    if isinstance(output, np.ndarray):
        if output.shape != tuple(img.shape):
            raise ValueError(f"output has shape {output.shape}, expected {tuple(img.shape)}")
        output[...] = convolution(img, scaling_function, s).cpu().numpy()
        return output
    if output is not None and not isinstance(output, torch.Tensor):
        raise TypeError("output must be a NumPy array or a torch tensor")
    if img.ndim == 2:
        out, _ = atrous_scale(img, s, scaling_function, out_c=output, out_w=False)
    else:
        out = _smooth_nd(img.contiguous(), int(s), scaling_function)
        if output is not None:
            output.copy_(out)
            out = output
    return out.cpu().numpy() if (was_numpy and output is None) else out


def _smooth_nd(arr, s, scaling_function):
    """S_s of a contiguous 1-D signal (mirror border, watroo/wavelets.py:64-69) or 3-D volume (2-D smooth of every
    slice, then the depth pass, :46-63, wb_atrous_scale_volume) -- one scale of AtrousTransform._run_nd without the
    detail plane."""
    if arr.ndim == 1:
        return _smooth_nd_reference(arr, s, scaling_function)
    lib = _lib.load(require_cuda=True)
    out = torch.empty_like(arr)
    tmp = torch.empty_like(arr)
    with torch.cuda.device(arr.device):
        _lib.check(lib.wb_atrous_scale_volume(arr.data_ptr(), out.data_ptr(), None, tmp.data_ptr(), *arr.shape, int(s),
                                              scaling_function.taps_code, _lib.dtype_code(arr.dtype),
                                              _lib.stream_ptr(arr.device)))
    return out


def _smooth_nd_reference(arr, s, scaling_function):
    """_smooth_nd on wb_atrous_scale + wb_atrous_axis (one thread per sample, taps gathered from global memory): the
    route the volume kernels are checked against."""
    lib = _lib.load(require_cuda=True)
    code, taps = _lib.dtype_code(arr.dtype), scaling_function.taps_code
    out = torch.empty_like(arr)
    with torch.cuda.device(arr.device):
        if arr.ndim == 1:
            _lib.check(lib.wb_atrous_axis(arr.data_ptr(), arr.data_ptr(), out.data_ptr(), 0, 1, arr.shape[0], 1, s, taps,
                                          code, _lib.WB_BORDER_MIRROR, _lib.stream_ptr(arr.device)))
        else:
            depth, h, w = arr.shape
            tmp, _ = atrous_scale(arr, s, scaling_function, out_w=False)  # every [i] slice, one launch
            _lib.check(lib.wb_atrous_axis(tmp.data_ptr(), arr.data_ptr(), out.data_ptr(), 0, 1, depth, h * w, s, taps,
                                          code, _lib.WB_BORDER_SYMMETRIC, _lib.stream_ptr(arr.device)))
    return out


def bilateral_list(bilateral, level):
    """watroo/wavelets.py:421-424: a scalar is broadcast to level+1 entries, a list is copied and padded with 1."""
    sb = copy.copy(bilateral) if type(bilateral) is list else [bilateral, ] * (level + 1)
    if len(sb) <= level:
        sb.extend([1, ] * (level - len(sb) + 1))
    return sb


# ---------------------------------------------------------------------------------------------------------------
# Device reductions
# ---------------------------------------------------------------------------------------------------------------
def abs_median_noise(plane, sigma_e0, out_noise=None):
    """MAD noise of one plane per frame, on the device: ``(median(|plane|) / 0.6745) / sigma_e0`` -> float64 tensor of
    shape (batch,).  ``plane`` is (H, W) or (B, H, W) with contiguous frames.  No host synchronisation."""
    lib = _lib.load(require_cuda=True)
    b, h, w, pitch, bstride = _frame_layout(plane)
    if pitch != w:
        plane = plane.contiguous()
        b, h, w, pitch, bstride = _frame_layout(plane)
    code = _lib.dtype_code(plane.dtype)
    ws = torch.empty(lib.wb_abs_median_workspace_bytes(code, b, h * w), dtype=torch.uint8, device=plane.device)
    if out_noise is None:
        out_noise = torch.empty(b, dtype=torch.float64, device=plane.device)
    with torch.cuda.device(plane.device):
        _lib.check(lib.wb_abs_median(plane.data_ptr(), h * w, b, bstride, code, 0, out_noise.data_ptr(),
                                     float(sigma_e0), ws.data_ptr(), ws.numel(), _lib.stream_ptr(plane.device)))
    return out_noise


def abs_median(plane, compact=True):
    """Exact ``np.median(np.abs(plane))`` per frame as a tensor of the plane dtype, shape (batch,).  ``compact=False``
    gives the kernel the selection state only (every pass streams the plane; same result, for tests / A-B timing)."""
    lib = _lib.load(require_cuda=True)
    b, h, w, pitch, bstride = _frame_layout(plane)
    if pitch != w:
        plane = plane.contiguous()
        b, h, w, pitch, bstride = _frame_layout(plane)
    code = _lib.dtype_code(plane.dtype)
    ws = torch.empty(lib.wb_abs_median_workspace_bytes(code, b, h * w if compact else 0), dtype=torch.uint8,
                     device=plane.device)
    out = torch.empty(b, dtype=plane.dtype, device=plane.device)
    with torch.cuda.device(plane.device):
        _lib.check(lib.wb_abs_median(plane.data_ptr(), h * w, b, bstride, code, out.data_ptr(), 0, 1.0,
                                     ws.data_ptr(), ws.numel(), _lib.stream_ptr(plane.device)))
    return out


def plane_moments(planes):
    """Population [mean, variance, std] (float64) of each contiguous 2-D plane of ``planes`` ((H,W) or (N,H,W))."""
    lib = _lib.load(require_cuda=True)
    b, h, w, pitch, bstride = _frame_layout(planes)
    if pitch != w:
        planes = planes.contiguous()
        b, h, w, pitch, bstride = _frame_layout(planes)
    ws = torch.empty(lib.wb_plane_moments_workspace_bytes(b), dtype=torch.uint8, device=planes.device)
    out = torch.empty((b, 3), dtype=torch.float64, device=planes.device)
    with torch.cuda.device(planes.device):
        _lib.check(lib.wb_plane_moments(planes.data_ptr(), h * w, b, bstride, _lib.dtype_code(planes.dtype),
                                        out.data_ptr(), ws.data_ptr(), _lib.stream_ptr(planes.device)))
    return out


def synthesis(planes, out=None):
    """``np.sum(planes, axis=0)`` in plane order and plane dtype, on the device.  (N,H,W) -> (H,W); (B,N,H,W) ->
    (B,H,W).  ``out``: optional contiguous device tensor of that shape and dtype to write into."""
    lib = _lib.load(require_cuda=True)
    if not planes.is_contiguous():
        planes = planes.contiguous()
    if planes.ndim == 3:
        n, h, w = planes.shape
        b, in_bs = 1, 0
        shape = (h, w)
    else:
        b, n, h, w = planes.shape
        in_bs = n * h * w
        shape = (b, h, w)
    if out is None:
        out = torch.empty(shape, dtype=planes.dtype, device=planes.device)
    elif tuple(out.shape) != shape or out.dtype != planes.dtype or out.device != planes.device or not out.is_contiguous():
        raise ValueError("synthesis(): out must be a contiguous device tensor of the summed shape and the plane dtype")
    with torch.cuda.device(planes.device):
        _lib.check(lib.wb_synthesis(planes.data_ptr(), n, h * w, h * w, b, in_bs, out.data_ptr(), h * w,
                                    _lib.dtype_code(planes.dtype), _lib.stream_ptr(planes.device)))
    return out


def broadcast_noise_map(noise, shape, dtype, device):
    """A per-pixel noise map (ndarray or tensor) as a contiguous device tensor of ``shape`` and the plane dtype,
    broadcast NumPy-style as the reference's array arithmetic does (``data / (sigma * noise * sigma_e)``).  Raises
    ValueError when it does not broadcast to ``shape``."""
    m = noise if isinstance(noise, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(noise))
    try:
        m = torch.broadcast_to(m, tuple(shape))
    except RuntimeError as exc:
        raise ValueError(f"a noise map of shape {tuple(noise.shape)} does not broadcast to the plane shape "
                         f"{tuple(shape)}") from exc
    return m.to(device=device, dtype=dtype).contiguous()


class _Noise:
    """How a threshold kernel receives the noise: host scalar, device scalar (float64) or per-pixel map."""

    __slots__ = ("host", "dev", "map")

    def __init__(self, host=0.0, dev=None, map_=None):
        self.host, self.dev, self.map = host, dev, map_

    @property
    def dev_ptr(self):
        return 0 if self.dev is None else self.dev.data_ptr()

    @property
    def map_ptr(self):
        return 0 if self.map is None else self.map.data_ptr()


class Coefficients:
    """Wavelet planes plus the metadata needed to threshold them (mirror of watroo/wavelets.py:108-149).

    ``data``: torch CUDA tensor ``(L+1, H, W)``; ``scaling_function``: instance; ``bilateral``: what the transform
    was run with (selects the sigma_e table); ``noise``: None until needed, then the MAD estimate (kept on the
    device; reading the attribute synchronises and returns a float), or whatever the caller assigned: a number or
    a per-pixel map (ndarray / tensor)."""

    def __init__(self, data, scaling_function, bilateral=None):
        self.data = data
        self.scaling_function = scaling_function
        self.bilateral = bilateral
        self._noise = None

    def __len__(self):
        return len(self.data)

    def __array__(self, dtype=None, copy=None):
        """Host copy, so that ``np.sum(coefficients, axis=0)`` of the README keeps working."""
        host = self.data.detach().cpu().numpy()
        return host if dtype is None else host.astype(dtype, copy=False)

    @property
    def sigma_e(self):
        return self.scaling_function.sigma_e(bilateral=self.bilateral)

    # -- noise ------------------------------------------------------------------------------------------------
    @property
    def noise(self):
        n = self._noise
        if isinstance(n, torch.Tensor) and n.numel() == 1 and n.dtype == torch.float64 and n.ndim <= 1:
            return np.float64(n.item())
        return n

    @noise.setter
    def noise(self, value):
        self._noise = value

    def get_noise(self):
        """MAD estimate ``median(|w_0|) / 0.6745 / sigma_e[0]`` (watroo/wavelets.py:126-127) as a float64 scalar.
        Computed on the device (exact median); this accessor synchronises to hand back a number."""
        return np.float64(self._estimate_noise().item())

    def _estimate_noise(self):
        plane = self.data[0]
        if plane.ndim != 2:  # 1-D signal / 3-D volume: one frame of numel() samples
            plane = plane.reshape(1, -1)
        return abs_median_noise(plane, self.sigma_e[0])

    def _noise_arg(self, sigma):
        """Resolve ``self.noise`` for a threshold kernel, estimating it lazily like the reference
        (watroo/wavelets.py:131-132).  Returns a _Noise."""
        if self._noise is None:
            self._noise = self._estimate_noise()
        n = self._noise
        if isinstance(n, torch.Tensor):
            if n.numel() == 1 and n.ndim <= 1:
                if n.is_cuda and n.dtype == torch.float64:
                    return _Noise(dev=n)
                return _Noise(host=float(n.item()))
            return _Noise(map_=broadcast_noise_map(n, self.data.shape[1:], self.data.dtype, self.data.device))
        if isinstance(n, np.ndarray):
            if n.ndim == 0:
                return _Noise(host=float(n))
            m = broadcast_noise_map(n, self.data.shape[1:], self.data.dtype, self.data.device)
            self._noise = m  # keep the device copy for the next scale
            return _Noise(map_=m)
        if isinstance(n, numbers.Number):
            return _Noise(host=float(n))
        raise TypeError(f"unsupported noise type {type(n)}")

    # -- thresholding -------------------------------------------------------------------------------------------
    def significance(self, sigma, scale, soft_threshold=True):
        """watroo/wavelets.py:129-143.  ``sigma == 0`` or scalar ``noise == 0`` -> ones (plane dtype); soft ->
        float64 tensor ``erf(|w_s / (sigma noise sigma_e[s])|)``; hard -> bool tensor ``|w_s| > sigma noise sigma_e[s]``
        compared in float64."""
        plane = self.data[scale]
        if sigma == 0:
            return torch.ones_like(self.data[0])
        nz = self._noise_arg(sigma)
        if nz.map is None and nz.dev is None and nz.host == 0:
            return torch.ones_like(self.data[0])
        lib = _lib.load(require_cuda=True)
        if not plane.is_contiguous():
            plane = plane.contiguous()
        out = torch.empty(plane.shape, dtype=torch.float64 if soft_threshold else torch.uint8, device=plane.device)
        with torch.cuda.device(plane.device):
            _lib.check(lib.wb_significance(plane.data_ptr(), plane.numel(), _lib.dtype_code(plane.dtype), float(sigma),
                                           float(self.sigma_e[scale]), nz.host, nz.dev_ptr, nz.map_ptr,
                                           1 if soft_threshold else 0, out.data_ptr(), _lib.stream_ptr(plane.device)))
        return out if soft_threshold else out.view(torch.bool)

    def denoise(self, sigma, weights=None, soft_threshold=True):
        """watroo/wavelets.py:145-149: ``c *= wgt * significance(sig, scl)`` in place for the first ``len(sigma)``
        planes (the residual plane is never touched unless ``sigma`` is that long).  Returns None."""
        if weights is None:
            weights = (1,) * len(sigma)
        lib = _lib.load(require_cuda=True)
        for scl, (sig, wgt) in enumerate(zip(sigma, weights)):
            if scl >= len(self.data):
                break
            self._denoise_plane(lib, scl, sig, wgt, soft_threshold)

    def _denoise_plane(self, lib, scl, sig, wgt, soft_threshold):
        plane = self.data[scl]
        mode = 0
        nz = _Noise()
        if sig != 0:
            nz = self._noise_arg(sig)
            mode = 1 if soft_threshold else 2
            if nz.map is None and nz.dev is None and nz.host == 0:
                mode = 0
        if mode == 0 and wgt == 1:
            return
        assert plane.is_contiguous()
        with torch.cuda.device(plane.device):
            _lib.check(lib.wb_denoise_plane(plane.data_ptr(), plane.numel(), 1, 0, _lib.dtype_code(plane.dtype), mode,
                                            float(sig), float(self.sigma_e[scl]), nz.host, nz.dev_ptr, nz.map_ptr,
                                            float(wgt), _lib.stream_ptr(plane.device)))


class AtrousTransform:
    """Dyadic 'à trous' transform (mirror of watroo/wavelets.py:290-328, standard algorithm :408-444)."""

    def __init__(self, scaling_function_class=B3spline, bilateral=None, bilateral_scaling=False):
        self.scaling_function_class = scaling_function_class
        self.bilateral = bilateral
        self.bilateral_scaling = bilateral_scaling

    def __call__(self, arr, level, recursive=False):
        """Transform an image over ``level`` scales -> ``Coefficients`` with ``level + 1`` planes.

        2-D images take the row-pipeline kernels.  3-D volumes (2-D smooth of every slice, then the depth pass,
        watroo/wavelets.py:46-63) run the plain cascade through ``wb_atrous_transform_volume``, 1-D signals
        (whole-sample 'mirror' border, watroo/wavelets.py:64-69) through ``wb_atrous_axis``, and both bilateral
        cascades through ``wb_atrous_scale_bilateral_nd``.

        ``recursive=True`` on a plain 2-D transform reproduces the RESULT of the reference's recursive algorithm
        (watroo/wavelets.py:330-406; it differs from the standard one near the borders: symmetric pad by
        ``(taps // 2) * 2**(level-1)``, then every scale reflects inside its decimated sub-arrays) through a parity
        kernel (``wb_atrous_scale_lattice`` / ``wb_atrous_scale_bilateral_lattice``), not its CPU-side recursion.  For
        1-D / 3-D inputs the flag is ignored and the standard algorithm runs."""
        img, _ = to_device_image(arr, ndim_ok=(1, 2, 3))
        scaling_function = self.scaling_function_class(img.ndim)
        if recursive and img.ndim == 2 and int(level) >= 1:
            planes = self._run_recursive(img, int(level), scaling_function)
        elif img.ndim == 2:
            planes = self._run(img, int(level), scaling_function)
        else:
            planes = self._run_nd(img, int(level), scaling_function)
        return Coefficients(planes, scaling_function, self.bilateral)

    def _run_recursive(self, img, level, scaling_function):
        """Planes of ``atrous_recursive`` (watroo/wavelets.py:330-406) for a 2-D transform (plain or bilateral), level >= 1."""
        lib = _lib.load(require_cuda=True)
        n_taps = len(scaling_function.coefficients_1d)
        hw = (n_taps // 2) * 2 ** (level - 1)
        h, w = img.shape
        # np.pad(arr, hw, mode='symmetric') (:394-395), any number of reflections
        def sym(n):
            i = torch.arange(-hw, n + hw, device=img.device)
            m = torch.remainder(i, 2 * n)
            return torch.where(m < n, m, 2 * n - 1 - m)
        cur = img[sym(h)][:, sym(w)].contiguous()
        hp, wp = cur.shape
        full = torch.empty((level + 1, hp, wp), dtype=img.dtype, device=img.device)
        code, taps = _lib.dtype_code(img.dtype), scaling_function.taps_code
        factors = self.var_factors(level) if self.bilateral is not None else None
        with torch.cuda.device(img.device):
            for s in range(level):
                nxt = full[level] if s == level - 1 else torch.empty_like(cur)
                if factors is None:
                    _lib.check(lib.wb_atrous_scale_lattice(cur.data_ptr(), nxt.data_ptr(), full[s].data_ptr(), hp, wp, wp,
                                                           wp, wp, s, taps, code, _lib.stream_ptr(img.device)))
                else:  # watroo/wavelets.py:371-378: variance and range-weighted gather per decimated sub-array
                    _lib.check(lib.wb_atrous_scale_bilateral_lattice(cur.data_ptr(), nxt.data_ptr(), full[s].data_ptr(), hp,
                                                                     wp, wp, wp, wp, s, taps, code, factors[s],
                                                                     _lib.stream_ptr(img.device)))
                cur = nxt
        return full[:, hw:hw + h, hw:hw + w].contiguous()

    def _run_nd(self, arr, level, scaling_function):
        """Plain cascade of a 1-D signal or a 3-D volume: planes ``(level + 1, *arr.shape)``.  A plain volume is one
        wb_atrous_transform_volume call; bilateral volumes and 1-D signals take _run_nd_reference."""
        if level < 0:
            raise ValueError("level must be >= 0")
        if arr.ndim != 3 or self.bilateral is not None:
            return self._run_nd_reference(arr, level, scaling_function)
        lib = _lib.load(require_cuda=True)
        arr = arr.contiguous()
        planes = torch.empty((level + 1,) + tuple(arr.shape), dtype=arr.dtype, device=arr.device)
        code = _lib.dtype_code(arr.dtype)
        scratch = torch.empty(lib.wb_volume_scratch_bytes(code, *arr.shape, level), dtype=torch.uint8, device=arr.device)
        with torch.cuda.device(arr.device):
            _lib.check(lib.wb_atrous_transform_volume(arr.data_ptr(), planes.data_ptr(), scratch.data_ptr(), *arr.shape,
                                                      level, scaling_function.taps_code, code,
                                                      _lib.stream_ptr(arr.device)))
        return planes

    def _run_nd_reference(self, arr, level, scaling_function):
        """The per-scale cascade of a 1-D signal or a 3-D volume on wb_atrous_axis / wb_atrous_scale_bilateral_nd (for
        volumes the route wb_atrous_transform_volume is checked against)."""
        if level < 0:
            raise ValueError("level must be >= 0")
        lib = _lib.load(require_cuda=True)
        arr = arr.contiguous()
        planes = torch.empty((level + 1,) + tuple(arr.shape), dtype=arr.dtype, device=arr.device)
        if level == 0:
            planes[0].copy_(arr)
            return planes
        code, taps = _lib.dtype_code(arr.dtype), scaling_function.taps_code
        scratch = [torch.empty_like(arr) for _ in range(2 if level > 1 else 0)]
        sf2 = self.scaling_function_class(2)
        tmp = torch.empty_like(arr) if arr.ndim == 3 else None
        src = arr
        factors = self.var_factors(level) if self.bilateral is not None else None
        with torch.cuda.device(arr.device):
            for s in range(level):
                dst_c = planes[level] if s == level - 1 else scratch[s & 1]
                if factors is not None:
                    # bilateral cascade of a signal / volume (watroo/wavelets.py:433-442 on n-D input): parity kernel
                    shape3 = (1, 1, arr.shape[0]) if arr.ndim == 1 else tuple(arr.shape)
                    _lib.check(lib.wb_atrous_scale_bilateral_nd(src.data_ptr(), dst_c.data_ptr(), planes[s].data_ptr(),
                                                                arr.ndim, *shape3, s, taps, code, factors[s],
                                                                _lib.stream_ptr(arr.device)))
                elif arr.ndim == 1:
                    _lib.check(lib.wb_atrous_axis(src.data_ptr(), src.data_ptr(), dst_c.data_ptr(), planes[s].data_ptr(),
                                                  1, arr.shape[0], 1, s, taps, code, _lib.WB_BORDER_MIRROR,
                                                  _lib.stream_ptr(arr.device)))
                else:
                    depth, h, w = arr.shape
                    atrous_scale(src, s, sf2, out_c=tmp, out_w=False)  # every [i] slice, one launch
                    _lib.check(lib.wb_atrous_axis(tmp.data_ptr(), src.data_ptr(), dst_c.data_ptr(), planes[s].data_ptr(),
                                                  1, depth, h * w, s, taps, code, _lib.WB_BORDER_SYMMETRIC,
                                                  _lib.stream_ptr(arr.device)))
                src = dst_c
        return planes

    def batch(self, frames, level):
        """NEW entry point (no reference equivalent): transform a stack ``(B, H, W)`` of independent frames with one
        launch per scale.  Returns a ``(B, level + 1, H, W)`` tensor."""
        stack, _ = to_device_image(frames, ndim_ok=(3,))
        return self._run(stack, int(level), self.scaling_function_class(2))

    def stream(self, frames, level, out=None, depth=2):
        """NEW entry point (no reference equivalent): transform a sequence of HOST frames ``(N, H, W)`` into a host
        array ``(N, level + 1, H, W)``, overlapping the host->device copy of frame n+1, the transform of frame n and
        the device->host copy of the planes of frame n-1 on three CUDA streams (``depth`` device buffers in flight).

        The per-frame cost of the plain call is dominated by PCIe (H*W in, (level+1)*H*W out); pipelining hides the
        upload and the kernels behind the download.  ``frames`` / ``out``: torch CPU tensors (pinned memory is used as
        is, pageable memory is staged through a pinned copy) or NumPy arrays; returns ``out`` (allocated pinned when
        None; a NumPy view of it for NumPy input).  Plain (non-bilateral) transforms only."""
        if self.bilateral is not None:
            raise NotImplementedError("stream() covers the plain cascade")
        was_numpy = not isinstance(frames, torch.Tensor)
        host = torch.from_numpy(np.ascontiguousarray(frames)) if was_numpy else frames
        if host.ndim != 3:
            raise ValueError("stream() takes a stack of frames (N, H, W)")
        if host.dtype not in (torch.float32, torch.float64):
            host = host.to(torch.float64)  # the reference's recast rule for integer inputs
        if host.is_cuda:
            raise ValueError("stream() takes host frames; use batch() for device-resident stacks")
        if not host.is_pinned():
            host = host.contiguous().pin_memory()
        level = int(level)
        n, h, w = host.shape
        if out is None:
            out = torch.empty((n, level + 1, h, w), dtype=host.dtype).pin_memory()
        out_t = torch.from_numpy(out) if isinstance(out, np.ndarray) else out
        if tuple(out_t.shape) != (n, level + 1, h, w) or out_t.dtype != host.dtype:
            raise ValueError("out must be (N, level + 1, H, W) of the frame dtype")
        staged = None
        if not out_t.is_pinned():
            staged = torch.empty(out_t.shape, dtype=out_t.dtype).pin_memory()
        dst = out_t if staged is None else staged
        lib = _lib.load(require_cuda=True)
        dev = _device()
        sf = self.scaling_function_class(2)
        code = _lib.dtype_code(host.dtype)
        depth = max(1, min(int(depth), n))
        s_in, s_cmp, s_out = (torch.cuda.Stream(dev) for _ in range(3))
        caller = torch.cuda.current_stream(dev)
        for st in (s_in, s_cmp, s_out):
            st.wait_stream(caller)
        d_in = [torch.empty((h, w), dtype=host.dtype, device=dev) for _ in range(depth)]
        d_pl = [torch.empty((level + 1, h, w), dtype=host.dtype, device=dev) for _ in range(depth)]
        scratch = torch.empty((2, h, w), dtype=host.dtype, device=dev) if level > 1 else None
        ev_in = [torch.cuda.Event() for _ in range(depth)]
        ev_cmp = [torch.cuda.Event() for _ in range(depth)]
        ev_out = [torch.cuda.Event() for _ in range(depth)]
        with torch.cuda.device(dev):
            for i in range(n):
                b = i % depth
                with torch.cuda.stream(s_in):
                    if i >= depth:
                        s_in.wait_event(ev_cmp[b])       # the transform that read d_in[b] is done
                    d_in[b].copy_(host[i], non_blocking=True)
                    ev_in[b].record(s_in)
                with torch.cuda.stream(s_cmp):
                    s_cmp.wait_event(ev_in[b])
                    if i >= depth:
                        s_cmp.wait_event(ev_out[b])      # the download of d_pl[b] is done
                    _lib.check(lib.wb_atrous_transform(
                        d_in[b].data_ptr(), d_pl[b].data_ptr(), 0 if scratch is None else scratch.data_ptr(), 1, h, w,
                        w, 0, level, sf.taps_code, code, s_cmp.cuda_stream))
                    ev_cmp[b].record(s_cmp)
                with torch.cuda.stream(s_out):
                    s_out.wait_event(ev_cmp[b])
                    dst[i].copy_(d_pl[b], non_blocking=True)
                    ev_out[b].record(s_out)
        for st in (s_in, s_cmp, s_out):
            caller.wait_stream(st)
        s_out.synchronize()  # the result lives in host memory: hand it back complete
        if staged is not None:
            out_t.copy_(staged)
        return out if (isinstance(out, np.ndarray) or not was_numpy) else out_t.numpy()

    # -- internals ----------------------------------------------------------------------------------------------
    def var_factors(self, level):
        """sigma_b[s]**2 * (s + 1 if bilateral_scaling) for s < level (watroo/wavelets.py:421-424, :434-436)."""
        sb = bilateral_list(self.bilateral, level)
        return [float(sb[s]) ** 2 * ((s + 1) if self.bilateral_scaling else 1) for s in range(level)]

    def _run(self, img, level, scaling_function):
        if level < 0:
            raise ValueError("level must be >= 0")
        lib = _lib.load(require_cuda=True)
        b, h, w, pitch, bstride = _frame_layout(img)
        batched = img.ndim == 3
        shape = (b, level + 1, h, w) if batched else (level + 1, h, w)
        planes = torch.empty(shape, dtype=img.dtype, device=img.device)
        if self.bilateral is None:
            scratch = torch.empty((2, b, h, w), dtype=img.dtype, device=img.device) if level > 1 else None
            with torch.cuda.device(img.device):
                _lib.check(lib.wb_atrous_transform(
                    img.data_ptr(), planes.data_ptr(), 0 if scratch is None else scratch.data_ptr(), b, h, w, pitch,
                    bstride, level, scaling_function.taps_code, _lib.dtype_code(img.dtype),
                    _lib.stream_ptr(img.device)))
            return planes
        # bilateral cascade: one fused K2 launch per scale, c_s ping-pong in scratch
        view = planes if batched else planes.unsqueeze(0)  # (B, L+1, H, W)
        if level == 0:
            view[:, 0].copy_(img if batched else img.unsqueeze(0))
            return planes
        factors = self.var_factors(level)
        scratch = torch.empty((2, b, h, w), dtype=img.dtype, device=img.device)
        src = img if batched else img.unsqueeze(0)
        for s in range(level):
            dst_c = view[:, level] if s == level - 1 else scratch[s & 1]
            atrous_scale(src, s, scaling_function, out_c=dst_c, out_w=view[:, s], var_factor=factors[s])
            src = dst_c
        return planes


def randn_field(shape, seed, offset=0, device=None):
    """fp32 N(0,1) field from the library's Philox generator (device stand-in for np.random.normal)."""
    lib = _lib.load(require_cuda=True)
    device = device or _device()
    out = torch.empty(shape, dtype=torch.float32, device=device)
    with torch.cuda.device(device):
        _lib.check(lib.wb_randn_f32(out.data_ptr(), out.numel(), int(seed), int(offset), _lib.stream_ptr(device)))
    return out


def noise_weights(scaling_function, n_scales, n_trials=100, bilateral=None, fields=None, seed=None):
    """compute_noise_weights (watroo/wavelets.py:221-229) on the device; see AbstractScalingFunction."""
    nd = scaling_function.n_dim
    transform = AtrousTransform(scaling_function.__class__, bilateral=bilateral)
    side = len(scaling_function.sigma_e_1d) * 2 ** n_scales
    if seed is None:
        seed = int(np.random.SeedSequence().entropy % (2 ** 63))
    total = torch.zeros(n_scales, dtype=torch.float64, device=_device())
    it = iter(fields) if fields is not None else None
    quads = (side ** nd + 3) // 4
    for trial in range(n_trials):
        if it is not None:
            field, _ = to_device_image(next(it), ndim_ok=(nd,))
        else:
            field = randn_field((side,) * nd, seed, offset=trial * quads)
        if nd == 2:
            planes = transform._run(field, n_scales, scaling_function)
            total += plane_moments(planes[:-1])[:, 2]
        else:  # 1-D signals / 3-D volumes: one "frame" of side**nd samples per plane
            planes = transform._run_nd(field, n_scales, scaling_function)
            total += plane_moments(planes[:-1].reshape(n_scales, 1, -1))[:, 2]
    return (total / n_trials).cpu().numpy()
