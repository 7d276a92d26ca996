"""Evaluation metrics of the reference harness on the device (SURVEY.md section 8f-2).

`experiments/experiment.py:436-463` converts `hr` and `sr.clip(0, 1)` (:746-748) to the Y channel of YCbCr
(`utils/utils.py:170-186`) and calls `skimage.metrics.peak_signal_noise_ratio(hr_y, sr_y, data_range=1)` on the CPU, image by
image.  `psnr_y` does the same arithmetic in one fused CUDA pass over the two batches (C ABI `hitsir_psnr_y`), so evaluation
never copies the SR images to the host.  `ssim_y` does the same for the second score, `skimage.metrics.structural_similarity(hr_y,
sr_y, data_range=1)` (:575-640), in one fused CUDA pass plus a fixed-order reduction (C ABI `hitsir_ssim_y`).  There is no CPU path.
"""
from __future__ import annotations

import ctypes

import torch

from . import _capi


def mse_y(sr: torch.Tensor, hr: torch.Tensor, clip: bool = True) -> torch.Tensor:
    """Per-image mean squared difference of the Y channels, float64 CUDA tensor of shape (B,)."""
    if sr.device.type != "cuda" or hr.device != sr.device:
        raise RuntimeError("mse_y / psnr_y expect CUDA tensors on the same device: there is no CPU path.")
    if sr.dim() != 4 or sr.shape[1] != 3 or sr.shape != hr.shape:
        raise ValueError(f"expected two (B,3,H,W) batches of the same shape, got {tuple(sr.shape)} and {tuple(hr.shape)}")
    sr = sr.contiguous().float()
    hr = hr.contiguous().float()
    B, _, H, W = sr.shape
    lib = _capi.load()
    with torch.cuda.device(sr.device):
        stream = torch.cuda.current_stream(sr.device).cuda_stream
        scratch = torch.empty(int(lib.hitsir_psnr_y_scratch_doubles(B, H, W)), dtype=torch.float64, device=sr.device)
        out = torch.empty(B, dtype=torch.float64, device=sr.device)
        _capi.check(lib.hitsir_psnr_y(ctypes.c_void_p(sr.data_ptr()), ctypes.c_void_p(hr.data_ptr()), B, H, W, 1 if clip else 0,
                                      ctypes.c_void_p(scratch.data_ptr()), ctypes.c_void_p(out.data_ptr()), ctypes.c_void_p(stream)))
    return out


def psnr_y(sr: torch.Tensor, hr: torch.Tensor, clip: bool = True) -> torch.Tensor:
    """Per-image Y-channel PSNR in dB (data_range = 1), float64 CUDA tensor of shape (B,); +inf for identical images like skimage."""
    return 10.0 * torch.log10(1.0 / mse_y(sr, hr, clip))


def ssim_y(sr: torch.Tensor, hr: torch.Tensor, clip: bool = True, gaussian_weights: bool = False,
           use_sample_covariance: bool = True) -> torch.Tensor:
    """Per-image mean SSIM of the Y channels, float64 CUDA tensor of shape (B,): skimage 0.24's
    `structural_similarity(hr_y, sr_y, data_range=1, gaussian_weights=..., use_sample_covariance=...)` with `sr` clipped to [0, 1]
    first when `clip`.  Uniform 7x7 window by default; `gaussian_weights=True` takes the 11x11 Gaussian window (sigma 1.5).
    `gaussian_weights=True, use_sample_covariance=False` is the setting of Wang et al. that most papers report."""
    if sr.device.type != "cuda" or hr.device != sr.device:
        raise RuntimeError("ssim_y expects CUDA tensors on the same device: there is no CPU path.")
    if sr.dim() != 4 or sr.shape[1] != 3 or sr.shape != hr.shape:
        raise ValueError(f"expected two (B,3,H,W) batches of the same shape, got {tuple(sr.shape)} and {tuple(hr.shape)}")
    win = 11 if gaussian_weights else 7
    B, _, H, W = sr.shape
    if B == 0:
        raise ValueError("ssim_y got an empty batch")
    if H < win or W < win:
        raise ValueError(f"ssim_y needs images of at least the {win}x{win} window, got {tuple(sr.shape)}")
    sr = sr.contiguous().float()
    hr = hr.contiguous().float()
    g = 1 if gaussian_weights else 0
    lib = _capi.load()
    with torch.cuda.device(sr.device):
        stream = torch.cuda.current_stream(sr.device).cuda_stream
        scratch = torch.empty(int(lib.hitsir_ssim_y_scratch_doubles(B, H, W, g)), dtype=torch.float64, device=sr.device)
        out = torch.empty(B, dtype=torch.float64, device=sr.device)
        _capi.check(lib.hitsir_ssim_y(ctypes.c_void_p(sr.data_ptr()), ctypes.c_void_p(hr.data_ptr()), B, H, W, 1 if clip else 0, g,
                                      1 if use_sample_covariance else 0, ctypes.c_void_p(scratch.data_ptr()),
                                      ctypes.c_void_p(out.data_ptr()), ctypes.c_void_p(stream)))
    return out


def to_uint8_hwc(y: torch.Tensor) -> torch.Tensor:
    """`to_pil_image(y.clip(0, 1))` of test_experiment.py:75-77 on the device: fp32 (B,C,H,W) -> uint8 (B,H,W,C), value * 255 truncated
    (C ABI `hitsir_f32nchw_to_u8hwc`).  The multi-GPU output gather moves this form: a quarter of the fp32 bytes."""
    if y.device.type != "cuda" or y.dim() != 4:
        raise RuntimeError("to_uint8_hwc expects a (B,C,H,W) CUDA tensor: there is no CPU path.")
    y = y.contiguous().float()
    B, C, H, W = y.shape
    out = torch.empty((B, H, W, C), dtype=torch.uint8, device=y.device)
    with torch.cuda.device(y.device):
        stream = torch.cuda.current_stream(y.device).cuda_stream
        _capi.check(_capi.load().hitsir_f32nchw_to_u8hwc(ctypes.c_void_p(y.data_ptr()), ctypes.c_void_p(out.data_ptr()), B, C, H, W,
                                                          ctypes.c_void_p(stream)))
    return out
