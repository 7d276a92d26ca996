"""ctypes binding of the C ABI declared in include/hitsir_b200.h.

This is the whole Python<->native boundary: plain pointers and sizes.  The library is built
in-tree by `build.py` (`__graft_entry__.build()`); if it is missing or stale this module raises
instead of falling back to anything else -- there is no CPU or PyTorch implementation of the path.
"""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

HITSIR_MAX_LAYERS = 16
HITSIR_MAX_DEPTH = 16

UPSAMPLERS = {None: 0, "": 0, "pixelshuffle": 1, "pixelshuffledirect": 2, "nearest+conv": 3}

ERR_CUDA, ERR_INVALID, ERR_UNSUPPORTED, ERR_INPUT_TOO_SMALL, ERR_WEIGHTS, ERR_WORKSPACE = 1, 2, 3, 4, 5, 6

RESIZE_PIL, RESIZE_MATLAB = 0, 1


class HitsirConfig(C.Structure):
    _fields_ = [
        ("is_mult_size_conv_feat_extract", C.c_int32),
        ("is_channel_spatial_attn", C.c_int32),
        ("is_fusion", C.c_int32),
        ("in_chans", C.c_int32),
        ("embed_dim", C.c_int32),
        ("num_layers", C.c_int32),
        ("depths", C.c_int32 * HITSIR_MAX_LAYERS),
        ("num_heads", C.c_int32 * HITSIR_MAX_LAYERS),
        ("base_win_size", C.c_int32 * 2),
        ("mlp_ratio", C.c_float),
        ("upscale", C.c_int32),
        ("img_range", C.c_float),
        ("upsampler", C.c_int32),
        ("num_ratios", C.c_int32),
        ("hier_win_ratios", C.c_float * HITSIR_MAX_DEPTH),
        ("resi_3conv", C.c_int32),
        ("ape_tokens", C.c_int32),
    ]


HALO_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_void_p)
ALLREDUCE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_void_p)


class HitsirBand(C.Structure):
    _fields_ = [("frame_h", C.c_int32), ("row0", C.c_int32), ("layout_h", C.c_int32), ("has_top", C.c_int32), ("has_bottom", C.c_int32),
                ("halo", HALO_FN), ("allreduce", ALLREDUCE_FN), ("ctx", C.c_void_p)]


SYMBOLS = {
    # name: (restype, argtypes)
    "hitsir_create": (C.c_int, [C.POINTER(HitsirConfig), C.POINTER(C.c_void_p)]),
    "hitsir_destroy": (None, [C.c_void_p]),
    "hitsir_num_params": (C.c_int, [C.c_void_p]),
    "hitsir_param_name": (C.c_char_p, [C.c_void_p, C.c_int]),
    "hitsir_param_numel": (C.c_int64, [C.c_void_p, C.c_int]),
    "hitsir_set_param": (C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "hitsir_finalize_weights": (C.c_int, [C.c_void_p, C.c_void_p]),
    "hitsir_workspace_bytes": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_size_t)]),
    "hitsir_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]),
    "hitsir_workspace_bytes_band": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_size_t)]),
    "hitsir_forward_band": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.POINTER(HitsirBand), C.c_void_p, C.c_size_t, C.c_void_p]),
    "hitsir_forward_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_size_t, C.c_void_p]),
    "hitsir_forward_u8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_size_t, C.c_void_p]),
    "hitsir_workspace_bytes_x8": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_size_t)]),
    "hitsir_forward_x8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]),
    "hitsir_forward_x8_u8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_size_t,
                                       C.c_void_p]),
    "hitsir_f32nchw_to_u8hwc": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "hitsir_f32nchw_to_u8hwc_round": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "hitsir_basicsr_metrics_scratch_doubles": (C.c_int64, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]),
    "hitsir_psnr_ssim_basicsr": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                           C.c_void_p, C.c_void_p]),
    "hitsir_psnr_y_scratch_doubles":(C.c_int64, [C.c_int, C.c_int, C.c_int]),
    "hitsir_psnr_y": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "hitsir_ssim_y_scratch_doubles": (C.c_int64, [C.c_int, C.c_int, C.c_int, C.c_int]),
    "hitsir_ssim_y": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                C.c_void_p]),
    "hitsir_u8hwc_to_f32nchw": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "hitsir_resize_scratch_bytes": (C.c_int64, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]),
    "hitsir_resize_u8_pil": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "hitsir_resize_f32_matlab": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_void_p, C.c_void_p]),
    "hitsir_set_tap": (C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p, C.c_int64, C.c_int]),
    "hitsir_set_inject": (C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p, C.c_int64]),
    "hitsir_get_bias_table": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int64, C.c_void_p]),
    "hitsir_last_launch_count": (C.c_int64, [C.c_void_p]),
    "hitsir_profile_enable": (C.c_int, [C.c_void_p, C.c_int]),
    "hitsir_profile_num_categories": (C.c_int, [C.c_void_p]),
    "hitsir_profile_get": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
    "hitsir_set_gemm_backend": (C.c_int, [C.c_void_p, C.c_char_p]),
    "hitsir_last_error": (C.c_char_p, []),
    "hitsir_version": (C.c_char_p, []),
}

_lib = None


class HitsirError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(message)
        self.status = status


def library_path() -> str:
    """The in-tree product library.  HITSIR_B200_LIB names another build of this library (a build.py variant for a kernel
    experiment, or an earlier commit's build for an A/B comparison); it is never a different backend."""
    return os.environ.get("HITSIR_B200_LIB") or _build.LIB


def load():
    """Load libhitsir_b200.so (once).  Raises ImportError when it is missing or older than its sources."""
    global _lib
    if _lib is not None:
        return _lib
    path = library_path()
    if not os.path.exists(path):
        raise ImportError(
            f"{path} not found: build the CUDA library first (python __graft_entry__.py build, needs nvcc). "
            "hitsir_b200 has no CPU/PyTorch fallback for the forward pass.")
    stamp = os.path.join(_build.BUILD, "stamp.txt")
    if path == _build.LIB and os.path.exists(stamp) and os.path.isdir(_build.CSRC):
        try:
            if open(stamp).read().strip() != _build._digest():
                raise ImportError(f"{path} is older than its sources in {_build.CSRC}: rebuild (python __graft_entry__.py build)")
        except OSError:
            pass
    lib = C.CDLL(path)
    for name, (restype, argtypes) in SYMBOLS.items():
        fn = getattr(lib, name)       # AttributeError if the library does not export a declared symbol
        fn.restype = restype
        fn.argtypes = argtypes
    _lib = lib
    return lib


def last_error() -> str:
    return load().hitsir_last_error().decode("utf-8", "replace")


def check(status: int):
    """Map a C status to the exception the reference would raise at the same point."""
    if status == 0:
        return
    msg = last_error()
    if status == ERR_INPUT_TOO_SMALL:
        raise RuntimeError(msg)                    # F.pad(..., 'reflect') RuntimeError, hit_sir_pro.py:672
    if status == ERR_UNSUPPORTED:
        raise NotImplementedError(msg)
    raise HitsirError(status, msg)
