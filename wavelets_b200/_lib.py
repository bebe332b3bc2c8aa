"""ctypes binding of libwavelets_b200.so (the C ABI of include/wavelets_b200.h).

There is deliberately NO fallback: if the CUDA library cannot be loaded, or no CUDA device is present, every
operation raises.  torch is used for device memory and streams only.
"""
from __future__ import annotations

import ctypes
import os
import threading

import numpy as np
import torch

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libwavelets_b200.so")

WB_F32, WB_F64 = 0, 1
WB_TRIANGLE, WB_B3SPLINE = 3, 5
WB_BORDER_SYMMETRIC, WB_BORDER_MIRROR = 0, 1
WB_ENOT_FUSABLE = -7
ABI_VERSION = 2

_lock = threading.Lock()
_lib = None

_c_int, _c_ll, _c_vp, _c_dbl = ctypes.c_int, ctypes.c_longlong, ctypes.c_void_p, ctypes.c_double
_c_ull, _c_sz = ctypes.c_ulonglong, ctypes.c_size_t

# name -> (restype, argtypes); must list every symbol declared in include/wavelets_b200.h
SIGNATURES = {
    "wb_abi_version": (_c_int, []),
    "wb_error_string": (ctypes.c_char_p, [_c_int]),
    "wb_atrous_scale_path": (_c_int, [_c_int, _c_int, _c_ll, _c_ll, _c_int, _c_int, _c_int, _c_vp, _c_vp, _c_vp]),
    "wb_atrous_scale": (_c_int, [_c_vp, _c_vp, _c_vp, _c_int, _c_int, _c_int, _c_ll, _c_ll, _c_ll, _c_ll, _c_ll,
                                 _c_ll, _c_int, _c_int, _c_int, _c_vp]),
    "wb_atrous_transform": (_c_int, [_c_vp, _c_vp, _c_vp, _c_int, _c_int, _c_int, _c_ll, _c_ll, _c_int, _c_int,
                                     _c_int, _c_vp]),
    "wb_atrous_scale_band": (_c_int, [_c_vp, _c_vp, _c_vp, _c_int, _c_int, _c_int, _c_ll, _c_ll, _c_ll, _c_ll, _c_ll,
                                      _c_ll, _c_ll, _c_int, _c_int, _c_int, _c_vp]),
    "wb_wow_whiten_scale_band": (_c_int, [_c_vp, _c_vp, _c_int, _c_int, _c_int, _c_ll, _c_ll, _c_ll, _c_ll, _c_ll, _c_int,
                                          _c_int, _c_int, _c_int, _c_dbl, _c_dbl, _c_dbl, _c_vp, _c_dbl, _c_vp]),
    "wb_atrous_scale_lattice": (_c_int, [_c_vp, _c_vp, _c_vp, _c_int, _c_int, _c_ll, _c_ll, _c_ll, _c_int, _c_int, _c_int,
                                         _c_vp]),
    "wb_atrous_scale_bilateral_band": (_c_int, [_c_vp, _c_vp, _c_vp, _c_int, _c_int, _c_int, _c_ll, _c_ll, _c_ll, _c_ll,
                                                _c_ll, _c_ll, _c_ll, _c_int, _c_int, _c_int, _c_dbl, _c_vp]),
    "wb_atrous_scale_bilateral_lattice": (_c_int, [_c_vp, _c_vp, _c_vp, _c_int, _c_int, _c_ll, _c_ll, _c_ll, _c_int, _c_int,
                                                   _c_int, _c_dbl, _c_vp]),
    "wb_atrous_scale_band_push": (_c_int, [_c_vp, _c_vp, _c_vp, _c_int, _c_int, _c_int, _c_ll, _c_ll, _c_ll, _c_ll,
                                           _c_ll, _c_ll, _c_ll, _c_vp, _c_int, _c_vp, _c_int, _c_int, _c_int, _c_int,
                                           _c_vp]),
    "wb_atrous_scale_band_p2p": (_c_int, [_c_vp, _c_vp, _c_int, _c_int, _c_vp, _c_vp, _c_int, _c_int, _c_ll, _c_ll, _c_ll,
                                          _c_int, _c_int, _c_int, _c_vp]),
    "wb_atrous_scale_bilateral": (_c_int, [_c_vp, _c_vp, _c_vp, _c_int, _c_int, _c_int, _c_ll, _c_ll, _c_ll, _c_ll,
                                           _c_ll, _c_ll, _c_int, _c_int, _c_int, _c_dbl, _c_vp]),
    "wb_atrous_scale_bilateral_nd": (_c_int, [_c_vp, _c_vp, _c_vp, _c_int, _c_ll, _c_ll, _c_ll, _c_int, _c_int, _c_int,
                                              _c_dbl, _c_vp]),
    "wb_wow_whiten_scale": (_c_int, [_c_vp, _c_vp, _c_int, _c_int, _c_int, _c_ll, _c_ll, _c_ll, _c_ll, _c_int, _c_int,
                                     _c_int, _c_int, _c_dbl, _c_dbl, _c_dbl, _c_vp, _c_dbl, _c_vp]),
    "wb_wow_whiten_scale_map": (_c_int, [_c_vp, _c_vp, _c_vp, _c_int, _c_int, _c_int, _c_ll, _c_ll, _c_ll, _c_ll, _c_ll,
                                         _c_ll, _c_int, _c_int, _c_int, _c_int, _c_dbl, _c_dbl, _c_dbl, _c_vp]),
    "wb_wow_scale_path": (_c_int, [_c_int, _c_int, _c_int, _c_ll, _c_ll, _c_ll, _c_int, _c_int, _c_int, _c_vp, _c_vp,
                                   _c_vp]),
    "wb_wow_scale": (_c_int, [_c_vp, _c_vp, _c_vp, _c_int, _c_int, _c_int, _c_ll, _c_ll, _c_ll, _c_ll, _c_ll, _c_ll,
                              _c_int, _c_int, _c_int, _c_int, _c_dbl, _c_dbl, _c_dbl, _c_vp, _c_dbl, _c_vp]),
    "wb_abs_median_workspace_bytes": (_c_sz, [_c_int, _c_int, _c_ll]),
    "wb_abs_median": (_c_int, [_c_vp, _c_ll, _c_int, _c_ll, _c_int, _c_vp, _c_vp, _c_dbl, _c_vp, _c_sz, _c_vp]),
    "wb_plane_moments_workspace_bytes": (_c_sz, [_c_int]),
    "wb_plane_moments": (_c_int, [_c_vp, _c_ll, _c_int, _c_ll, _c_int, _c_vp, _c_vp, _c_vp]),
    "wb_significance": (_c_int, [_c_vp, _c_ll, _c_int, _c_dbl, _c_dbl, _c_dbl, _c_vp, _c_vp, _c_int, _c_vp, _c_vp]),
    "wb_denoise_plane": (_c_int, [_c_vp, _c_ll, _c_int, _c_ll, _c_int, _c_int, _c_dbl, _c_dbl, _c_dbl, _c_vp, _c_vp,
                                  _c_dbl, _c_vp]),
    "wb_residual_rescale": (_c_int, [_c_vp, _c_ll, _c_int, _c_ll, _c_int, _c_vp, _c_dbl, _c_vp]),
    "wb_synthesis": (_c_int, [_c_vp, _c_int, _c_ll, _c_ll, _c_int, _c_ll, _c_vp, _c_ll, _c_int, _c_vp]),
    "wb_randn_f32": (_c_int, [_c_vp, _c_ll, _c_ull, _c_ull, _c_vp]),
    "wb_wow_cascade_workspace_bytes": (_c_sz, [_c_int, _c_int, _c_ll]),
    "wb_wow_cascade": (_c_int, [_c_vp, _c_ll, _c_ll, _c_vp, _c_vp, _c_vp, _c_int, _c_int, _c_int, _c_int, _c_int, _c_int,
                                ctypes.POINTER(_c_dbl), ctypes.POINTER(_c_dbl), ctypes.POINTER(_c_dbl),
                                ctypes.POINTER(_c_dbl), _c_int, _c_dbl, _c_vp, _c_int, _c_vp, _c_sz, _c_vp]),
    "wb_wow_cascade_map": (_c_int, [_c_vp, _c_ll, _c_ll, _c_vp, _c_vp, _c_vp, _c_int, _c_int, _c_int, _c_int, _c_int,
                                    _c_int, ctypes.POINTER(_c_dbl), ctypes.POINTER(_c_dbl), ctypes.POINTER(_c_dbl),
                                    ctypes.POINTER(_c_dbl), _c_int, _c_vp, _c_ll, _c_ll, _c_vp, _c_sz, _c_vp]),
    "wb_wow_cascade_blend_workspace_bytes": (_c_sz, [_c_int, _c_int, _c_ll]),
    "wb_wow_cascade_blend": (_c_int, [_c_vp, _c_ll, _c_ll, _c_vp, _c_vp, _c_vp, _c_vp, _c_int, _c_int, _c_int, _c_int,
                                      _c_int, _c_int, ctypes.POINTER(_c_dbl), ctypes.POINTER(_c_dbl),
                                      ctypes.POINTER(_c_dbl), ctypes.POINTER(_c_dbl), _c_int, _c_dbl, _c_vp, _c_int,
                                      _c_int, _c_vp, _c_ll, _c_ll, _c_int, _c_int, _c_dbl, _c_dbl, _c_dbl, _c_int, _c_dbl,
                                      _c_int, _c_vp, _c_sz, _c_vp]),
    "wb_filter2d": (_c_int, [_c_vp, _c_vp, _c_int, _c_int, _c_ll, _c_ll, _c_vp, _c_int, _c_int, _c_int, _c_int, _c_vp]),
    "wb_atrous_axis": (_c_int, [_c_vp, _c_vp, _c_vp, _c_vp, _c_ll, _c_ll, _c_ll, _c_int, _c_int, _c_int, _c_int, _c_vp]),
    "wb_atrous_scale_volume": (_c_int, [_c_vp, _c_vp, _c_vp, _c_vp, _c_int, _c_int, _c_int, _c_int, _c_int, _c_int,
                                        _c_vp]),
    "wb_volume_scratch_bytes": (_c_sz, [_c_int, _c_int, _c_int, _c_int, _c_int]),
    "wb_atrous_transform_volume": (_c_int, [_c_vp, _c_vp, _c_vp, _c_int, _c_int, _c_int, _c_int, _c_int, _c_int, _c_vp]),
    "wb_wow_cascade_volume_workspace_bytes": (_c_sz, [_c_int, _c_int, _c_int, _c_int]),
    "wb_wow_cascade_volume": (_c_int, [_c_vp, _c_vp, _c_vp, _c_vp, _c_int, _c_int, _c_int, _c_int, _c_int, _c_int,
                                       ctypes.POINTER(_c_dbl), ctypes.POINTER(_c_dbl), ctypes.POINTER(_c_dbl), _c_int,
                                       _c_int, _c_dbl, _c_vp, _c_int, _c_vp, _c_ll, _c_vp, _c_sz, _c_vp]),
}
# development hooks exported by the library but not part of the stable ABI
_EXTRA = {
    "wb_tune_k1": (_c_int, [_c_int, _c_int, _c_int, _c_int, _c_int]),
}


def load(require_cuda: bool = False) -> ctypes.CDLL:
    """Load the shared library (once).  Raises RuntimeError when it is missing -- there is no CPU path."""
    global _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise RuntimeError(
                    f"{LIB_PATH} is missing: build it with `python -m wavelets_b200.build` "
                    "(wavelets_b200 has no CPU fallback)")
            lib = ctypes.CDLL(LIB_PATH)
            for name, (res, args) in {**SIGNATURES, **_EXTRA}.items():
                fn = getattr(lib, name)
                fn.restype, fn.argtypes = res, args
            if lib.wb_abi_version() != ABI_VERSION:
                raise RuntimeError("libwavelets_b200.so ABI version mismatch; rebuild it")
            _lib = lib
    if require_cuda and not torch.cuda.is_available():
        raise RuntimeError("wavelets_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    return _lib


def check(status: int) -> None:
    if status != 0:
        msg = load().wb_error_string(status).decode()
        raise RuntimeError(f"wavelets_b200: {msg} (status {status})")


def dtype_code(dtype: torch.dtype) -> int:
    if dtype == torch.float32:
        return WB_F32
    if dtype == torch.float64:
        return WB_F64
    raise TypeError(f"wavelets_b200 computes in float32 or float64, got {dtype}")


def stream_ptr(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def np_to_torch_dtype(dt: np.dtype) -> torch.dtype:
    return {np.dtype(np.float32): torch.float32, np.dtype(np.float64): torch.float64}[np.dtype(dt)]
