"""Bicubic resizing and end-to-end scoring of HR images on the device (SURVEY.md section 8f-2: eval never leaves the device).

The reference's test stage (`experiments/experiment.py:660-790`) synthesises each LR input by bicubic downscaling on the CPU
(`datasets/dataset.py:51-91`), runs `model(lr).clip(0, 1)` and scores Y-channel PSNR / SSIM.  `resize_bicubic` does the downscaling
in CUDA (C ABI `hitsir_resize_u8_pil` / `hitsir_resize_f32_matlab`) in either standard definition:

* ``kernel="pil"``: Pillow 12.2's ``Image.resize((W, H), Image.BICUBIC)`` on uint8 images, bit for bit;
* ``kernel="matlab"``: MATLAB ``imresize(x, scale, 'bicubic')`` as BasicSR's ``imresize`` computes it (the copy at
  ``utils/utils.py:399-570``), fp32, within a derived bound of the fp64 result.

`evaluate` composes it with `to_float_nchw`, the model's forward and the metrics.  There is no CPU path.
"""
from __future__ import annotations

import ctypes
import math
from typing import Dict, Optional, Sequence

import torch

from . import _capi
from .metrics import psnr_ssim_basicsr, psnr_y, ssim_y, to_uint8_hwc


def to_float_nchw(x_u8: torch.Tensor) -> torch.Tensor:
    """torchvision's `to_tensor` of a uint8 (B,H,W,C) CUDA batch (utils/utils.py:143-145: value / 255) -> fp32 (B,C,H,W), on the
    device (C ABI `hitsir_u8hwc_to_f32nchw`, the conversion `forward_uint8` applies).  The mirror of `to_uint8_hwc`."""
    if x_u8.device.type != "cuda" or x_u8.dtype != torch.uint8 or x_u8.dim() != 4:
        raise RuntimeError("to_float_nchw expects a (B,H,W,C) uint8 CUDA tensor: there is no CPU path.")
    x_u8 = x_u8.contiguous()
    B, H, W, C = x_u8.shape
    out = torch.empty((B, C, H, W), dtype=torch.float32, device=x_u8.device)
    with torch.cuda.device(x_u8.device):
        stream = torch.cuda.current_stream(x_u8.device).cuda_stream
        _capi.check(_capi.load().hitsir_u8hwc_to_f32nchw(ctypes.c_void_p(x_u8.data_ptr()), ctypes.c_void_p(out.data_ptr()), B, C, H, W,
                                                          ctypes.c_void_p(stream)))
    return out


def resize_bicubic(x: torch.Tensor, size: Optional[Sequence[int]] = None, scale: Optional[float] = None,
                   kernel: str = "pil") -> torch.Tensor:
    """Bicubic resize of a CUDA batch.

    * ``kernel="pil"``: `x` uint8 (B,H,W,C), C in {1, 3}, ``size=(outH, outW)`` -> uint8 (B,outH,outW,C), equal bit for bit to
      Pillow's ``Image.resize((outW, outH), Image.BICUBIC)`` of each image (modes "L" / "RGB").
    * ``kernel="matlab"``: `x` fp32 (B,C,H,W), C in {1, 3}, `scale` > 0 -> fp32 (B,C,ceil(H*scale),ceil(W*scale)): MATLAB
      ``imresize(x, scale, 'bicubic')`` (antialiased when downscaling), values not clipped.
    """
    if kernel not in ("pil", "matlab"):
        raise ValueError(f"resize_bicubic: kernel must be 'pil' or 'matlab', got {kernel!r}")
    if x.device.type != "cuda" or x.dim() != 4:
        raise RuntimeError("resize_bicubic expects a 4-D CUDA tensor: there is no CPU path.")
    lib = _capi.load()
    if kernel == "pil":
        if x.dtype != torch.uint8:
            raise ValueError(f"resize_bicubic(kernel='pil') takes uint8 (B,H,W,C) images, got {x.dtype}")
        if size is None or scale is not None or len(size) != 2:
            raise ValueError("resize_bicubic(kernel='pil') takes size=(outH, outW) and no scale")
        B, H, W, C = x.shape
        outH, outW = int(size[0]), int(size[1])
        if C not in (1, 3) or B == 0 or H == 0 or W == 0 or outH <= 0 or outW <= 0:
            raise ValueError(f"resize_bicubic(kernel='pil'): bad shape {tuple(x.shape)} -> {(outH, outW)}")
        out = torch.empty((B, outH, outW, C), dtype=torch.uint8, device=x.device)
        mode = _capi.RESIZE_PIL
    else:
        if x.dtype != torch.float32:
            raise ValueError(f"resize_bicubic(kernel='matlab') takes float32 (B,C,H,W) images, got {x.dtype}")
        if scale is None or size is not None:
            raise ValueError("resize_bicubic(kernel='matlab') takes scale and no size")
        scale = float(scale)
        B, C, H, W = x.shape
        if C not in (1, 3) or B == 0 or H == 0 or W == 0 or not (scale > 0 and math.isfinite(scale)):
            raise ValueError(f"resize_bicubic(kernel='matlab'): bad shape {tuple(x.shape)} or scale {scale}")
        outH, outW = math.ceil(H * scale), math.ceil(W * scale)      # BasicSR's output size, the same double product as the C entry
        out = torch.empty((B, C, outH, outW), dtype=torch.float32, device=x.device)
        mode = _capi.RESIZE_MATLAB
    x = x.contiguous()
    with torch.cuda.device(x.device):
        stream = torch.cuda.current_stream(x.device).cuda_stream
        scratch = torch.empty(int(lib.hitsir_resize_scratch_bytes(mode, H, W, outH, outW)), dtype=torch.uint8, device=x.device)
        src, dst, scr = ctypes.c_void_p(x.data_ptr()), ctypes.c_void_p(out.data_ptr()), ctypes.c_void_p(scratch.data_ptr())
        if kernel == "pil":
            _capi.check(lib.hitsir_resize_u8_pil(src, dst, B, H, W, C, outH, outW, scr, ctypes.c_void_p(stream)))
        else:
            _capi.check(lib.hitsir_resize_f32_matlab(src, dst, B, C, H, W, scale, scr, ctypes.c_void_p(stream)))
    return out


def evaluate(model, hr_u8: torch.Tensor, lr_kernel: str = "pil", self_ensemble: bool = False, bicubic_baseline: bool = False,
             gaussian_weights: Optional[bool] = None, use_sample_covariance: Optional[bool] = None, protocol: str = "skimage",
             crop_border: Optional[int] = None, lr_u8: Optional[torch.Tensor] = None) -> Dict[str, torch.Tensor]:
    """Score `model` on a batch of HR images without leaving the device: the loop of experiments/experiment.py:681-790.

    `hr_u8`: uint8 (B,H,W,3) CUDA images, H and W multiples of ``model.upscale`` (crop by slicing first).  HR is
    ``to_float_nchw(hr_u8)``; the LR is the Pillow resize of `hr_u8` converted the same way (``lr_kernel="pil"``) or
    ``resize_bicubic(hr, scale=1/upscale, kernel="matlab")`` kept in fp32 (``lr_kernel="matlab"``); or, when given, `lr_u8`: uint8
    (B,H/upscale,W/upscale,3) LR images such as the MATLAB-made ones benchmark sets ship, converted by ``to_float_nchw``.  SR is
    ``model(lr)`` (or ``model.forward_x8(lr)``).  With `bicubic_baseline`, the LR is also upscaled back to H x W by the `lr_kernel`
    bicubic and scored the same way.

    ``protocol="skimage"`` (the reference harness): SR clipped to [0, 1] by the metrics, ``psnr_y`` and ``ssim_y`` with
    `gaussian_weights` / `use_sample_covariance` (default False / True).  ``protocol="basicsr"`` (published SR tables):
    ``to_uint8_hwc(sr, rounding="nearest")`` scored by ``psnr_ssim_basicsr(., hr_u8, crop_border, test_y_channel=True)``,
    `crop_border` defaulting to ``upscale``.  Returns ``{"psnr_y", "ssim_y"}``, float64 (B,) CUDA tensors, plus
    ``"bicubic_psnr_y"`` / ``"bicubic_ssim_y"`` with `bicubic_baseline`."""
    if lr_kernel not in ("pil", "matlab"):
        raise ValueError(f"evaluate: lr_kernel must be 'pil' or 'matlab', got {lr_kernel!r}")
    if protocol not in ("skimage", "basicsr"):
        raise ValueError(f"evaluate: protocol must be 'skimage' or 'basicsr', got {protocol!r}")
    if protocol == "basicsr" and (gaussian_weights is not None or use_sample_covariance is not None):
        raise ValueError("evaluate: gaussian_weights / use_sample_covariance are skimage options; protocol='basicsr' fixes its window")
    if protocol == "skimage" and crop_border is not None:
        raise ValueError("evaluate: crop_border applies to protocol='basicsr' only; the skimage protocol scores the whole image")
    if hr_u8.device.type != "cuda" or hr_u8.dtype != torch.uint8 or hr_u8.dim() != 4 or hr_u8.shape[3] != 3:
        raise ValueError(f"evaluate expects uint8 (B,H,W,3) CUDA images, got {hr_u8.dtype} {tuple(hr_u8.shape)} on {hr_u8.device}")
    s = int(model.upscale)
    if model.out_scale != s:
        raise ValueError("evaluate needs a super-resolution model (an upsampler): its output must be `upscale` times the input")
    B, H, W, _ = hr_u8.shape
    if H % s or W % s:
        raise ValueError(f"evaluate: H and W must be multiples of upscale={s}, got {H} x {W}; crop the HR images first")
    c = s if crop_border is None else int(crop_border)
    if protocol == "basicsr" and (c < 0 or H - 2 * c < 11 or W - 2 * c < 11):
        raise ValueError(f"evaluate: crop_border={c} leaves less than the 11x11 SSIM window of {H} x {W} images")
    hr = to_float_nchw(hr_u8)
    if lr_u8 is not None:
        if lr_u8.dtype != torch.uint8 or lr_u8.device != hr_u8.device or tuple(lr_u8.shape) != (B, H // s, W // s, 3):
            raise ValueError(f"evaluate: lr_u8 must be uint8 {(B, H // s, W // s, 3)} on {hr_u8.device}, got {lr_u8.dtype} "
                             f"{tuple(lr_u8.shape)} on {lr_u8.device}")
        lr = to_float_nchw(lr_u8)
    elif lr_kernel == "pil":
        lr_u8 = resize_bicubic(hr_u8, size=(H // s, W // s), kernel="pil")
        lr = to_float_nchw(lr_u8)
    else:
        lr = resize_bicubic(hr, scale=1.0 / s, kernel="matlab")
    with torch.no_grad():
        sr = model.forward_x8(lr) if self_ensemble else model(lr)
    if protocol == "skimage":
        kw = dict(gaussian_weights=bool(gaussian_weights), use_sample_covariance=use_sample_covariance is None or bool(use_sample_covariance))
        score = lambda y: (psnr_y(y, hr), ssim_y(y, hr, **kw))     # noqa: E731
    else:
        score = lambda y: psnr_ssim_basicsr(to_uint8_hwc(y, rounding="nearest"), hr_u8, c, test_y_channel=True)     # noqa: E731
    out = dict(zip(("psnr_y", "ssim_y"), score(sr)))
    if bicubic_baseline:
        if lr_kernel == "pil":
            up = to_float_nchw(resize_bicubic(lr_u8, size=(H, W), kernel="pil"))
        else:
            up = resize_bicubic(lr, scale=float(s), kernel="matlab")
        out["bicubic_psnr_y"], out["bicubic_ssim_y"] = score(up)
    return out
