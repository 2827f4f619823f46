"""ctypes binding of ``libcistaflow.so`` (C ABI: ``include/cistaflow.h``).

The library is the product; this module only marshals pointers.  There is NO
CPU fallback: if the shared library is missing, or the current device is not a
B200-class (sm_100) GPU, every op raises ``RuntimeError``.
"""
from __future__ import annotations

import ctypes
import os
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CISTAFLOW_LIB", os.path.join(_HERE, "libcistaflow.so"))

# enums of include/cistaflow.h
VOXEL_ATOMIC, VOXEL_DETERMINISTIC, VOXEL_ATOMIC_L2, VOXEL_ATOMIC_TILED = 0, 1, 2, 3
FLAVOUR_TORCH, FLAVOUR_NUMPY, FLAVOUR_POL, FLAVOUR_MVSEC = 0, 1, 2, 3
PRE_NONE, PRE_STD, PRE_MAXMIN = 0, 1, 2
WINDOWS_FIXED, WINDOWS_SPLIT = 0, 1
CORR_TF32, CORR_FP32, CORR_3XTF32, CORR_F16, CORR_AUTO = 0, 1, 2, 3, 4
CORR_MAX_LEVELS = 6

STATUS = {0: "CF_OK", -1: "CF_ERR_INVALID_ARG", -2: "CF_ERR_NULL", -3: "CF_ERR_ALIGN", -4: "CF_ERR_ARCH",
          -5: "CF_ERR_WORKSPACE", -6: "CF_ERR_CUDA", -7: "CF_ERR_UNSUPPORTED"}

# every symbol include/cistaflow.h declares: (restype, argtypes)
_vp, _i, _i64, _f, _sz = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_float, ctypes.c_size_t
SYMBOLS = {
    "cf_version": (_i, []),
    "cf_last_error": (ctypes.c_char_p, []),
    "cf_device_check": (_i, []),
    "cf_launch_count": (_i64, []),
    "cf_last_kernel": (ctypes.c_char_p, []),
    "cf_voxel_workspace_bytes": (_sz, [_i64, _i, _i, _i, _i, _i, _i, _i]),
    "cf_voxel_bin": (_i, [_vp, _vp, _i64, _i, _i, _i, _i, _i, _i, _i, _f, _vp, _vp, _sz, _vp]),
    "cf_preprocess_workspace_bytes": (_sz, [_i, _i64]),
    "cf_voxel_preprocess": (_i, [_vp, _vp, _i, _i64, _i, _f, _vp, _sz, _vp]),
    "cf_events_pack": (_i, [_vp, _vp, _i64, _i, _vp, _vp]),
    "cf_events_filter_workspace_bytes": (_sz, [_i64]),
    "cf_events_filter": (_i, [_vp, _i64, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    "cf_event_window_offsets": (_i, [_vp, _i, _i64, _vp, _i, _vp, _vp]),
    "cf_voxel_bin_packed": (_i, [_vp, _vp, _i64, _i, _i, _i, _i, _i, _f, _vp, _vp, _sz, _vp]),
    "cf_warp": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _f, _vp]),
    "cf_warp_frame_and_codes": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _f, _vp]),
    "cf_flow_any": (_i, [_vp, _i64, _vp, _vp]),
    "cf_warp_frame_and_codes_gated": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _f, _vp, _vp]),
    "cf_warp_frame_and_codes_upflow8": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _f, _vp]),
    "cf_warp_backward": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _f, _vp]),
    "cf_voxel_flow_warp_workspace_bytes": (_sz, [_i, _i, _i]),
    "cf_voxel_flow_warp": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    "cf_corr_workspace_bytes": (_sz, [_i, _i, _i, _i, _i, _i]),
    "cf_corr_build": (_i, [_vp, _vp, _i, _i, _i, _i, _i, ctypes.POINTER(_vp), _i, _vp, _sz, _vp]),
    "cf_corr_lookup": (_i, [ctypes.POINTER(_vp), _vp, _i, _i, _i, _i, _i, _vp, _vp]),
    "cf_corr_lookup_backward": (_i, [_vp, ctypes.POINTER(_vp), _vp, _i, _i, _i, _i, _i, ctypes.POINTER(_vp), _vp, _vp]),
}
# every symbol include/cistaflow_altcorr.h declares (the on-demand correlation lookup, compiled into the same library)
ALTCORR_SYMBOLS = {
    "cf_corr_alt_workspace_bytes": (_sz, [_i, _i, _i, _i, _i, _i]),
    "cf_corr_alt_prepare": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _sz, _vp]),
    "cf_corr_alt_lookup": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp, _vp]),
}
# every symbol include/cistaflow_det.h declares (the deterministic warp adjoint, compiled into the same library)
DET_SYMBOLS = {
    "cf_warp_backward_det_workspace_bytes": (_sz, [_i, _i, _i, _i, _i, _i]),
    "cf_warp_backward_det": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _f, _vp, _sz, _vp]),
}

# every symbol include/cistaflow_half.h declares (the opt-in fp16 correlation pyramid, compiled into the same library)
HALF_SYMBOLS = {
    "cf_corr_build_half": (_i, [_vp, _vp, _i, _i, _i, _i, _i, ctypes.POINTER(_vp), _i, _vp, _sz, _vp]),
    "cf_corr_lookup_half": (_i, [ctypes.POINTER(_vp), _vp, _i, _i, _i, _i, _i, _vp, _vp]),
}

_lock = threading.Lock()
_lib = None


class CistaFlowError(RuntimeError):
    """A libcistaflow entry point returned a negative cf_status."""


def load() -> ctypes.CDLL:
    """dlopen the library and bind every symbol of the four headers (no GPU needed)."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise RuntimeError(
                    f"libcistaflow.so not found at {LIB_PATH}: build it with "
                    f"`python cista-flow_b200/build.py` (or __graft_entry__.build()). "
                    f"There is no CPU / PyTorch fallback for the hot path.")
            lib = ctypes.CDLL(LIB_PATH)
            for name, (res, args) in {**SYMBOLS, **ALTCORR_SYMBOLS, **DET_SYMBOLS, **HALF_SYMBOLS}.items():
                fn = getattr(lib, name)  # AttributeError if the .so lacks a declared symbol
                fn.restype, fn.argtypes = res, args
            _lib = lib
    return _lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().cf_last_error().decode(errors="replace")
        exc = ValueError if rc in (-1, -2, -3) else CistaFlowError
        raise exc(f"{what}: {STATUS.get(rc, rc)}: {msg}")


def require_cuda(t: torch.Tensor, name: str) -> None:
    if not t.is_cuda:
        raise RuntimeError(f"{name} must live on a CUDA device (got {t.device}); "
                           f"the cistaflow hot path has no CPU fallback")


def stream_ptr(device: torch.device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def workspace(nbytes: int, device: torch.device) -> torch.Tensor | None:
    """Scratch from the torch caching allocator (stream-ordered reuse is safe)."""
    if nbytes <= 0:
        return None
    return torch.empty(nbytes, dtype=torch.uint8, device=device)


def ptr(t: torch.Tensor | None) -> int | None:
    return None if t is None else t.data_ptr()


def pointer_array(tensors) -> ctypes.Array:
    arr = (ctypes.c_void_p * len(tensors))()
    for k, t in enumerate(tensors):
        arr[k] = t.data_ptr()
    return arr
