"""Evaluation metrics of the reference harness on the device (SURVEY.md section 8f-2).

`experiments/experiment.py:436-463` converts `hr` and `sr.clip(0, 1)` (:746-748) to the Y channel of YCbCr
(`utils/utils.py:170-186`) and calls `skimage.metrics.peak_signal_noise_ratio(hr_y, sr_y, data_range=1)` on the CPU, image by
image.  `psnr_y` does the same arithmetic in one fused CUDA pass over the two batches (C ABI `hitsir_psnr_y`), so evaluation
never copies the SR images to the host.  `ssim_y` does the same for the second score, `skimage.metrics.structural_similarity(hr_y,
sr_y, data_range=1)` (:575-640), in one fused CUDA pass plus a fixed-order reduction (C ABI `hitsir_ssim_y`).  `psnr_ssim_basicsr`
scores by the other convention, BasicSR's `calculate_psnr` / `calculate_ssim` on rounded uint8 images, which published SR tables use.
There is no CPU path.
"""
from __future__ import annotations

import ctypes

import torch

from . import _capi


def _check_pair(sr: torch.Tensor, hr: torch.Tensor, who: str, u8_hwc: bool = False) -> None:
    """Raise unless `sr` and `hr` are CUDA tensors on one device with one shape: (B,3,H,W), or (B,H,W,3) and uint8 when `u8_hwc`.
    `who` names the caller and its verb in the device error ("ssim_y expects")."""
    if sr.device.type != "cuda" or hr.device != sr.device:
        raise RuntimeError(f"{who} CUDA tensors on the same device: there is no CPU path.")
    if u8_hwc and (sr.dtype != torch.uint8 or hr.dtype != torch.uint8):
        raise ValueError(f"{who.split()[0]} takes uint8 images, got {sr.dtype} and {hr.dtype}")
    layout, c = ("(B,H,W,3)", 3) if u8_hwc else ("(B,3,H,W)", 1)
    if sr.dim() != 4 or sr.shape[c] != 3 or sr.shape != hr.shape:
        raise ValueError(f"expected two {layout} batches of the same shape, got {tuple(sr.shape)} and {tuple(hr.shape)}")


def _call(fn, device: torch.device, *args) -> None:
    """Call the C ABI function `fn` on `device`, tensors passed by address and the current stream of `device` as the last argument."""
    with torch.cuda.device(device):
        stream = torch.cuda.current_stream(device).cuda_stream
        _capi.check(fn(*[ctypes.c_void_p(a.data_ptr()) if isinstance(a, torch.Tensor) else a for a in args], ctypes.c_void_p(stream)))


def mse_y(sr: torch.Tensor, hr: torch.Tensor, clip: bool = True) -> torch.Tensor:
    """Per-image mean squared difference of the Y channels, float64 CUDA tensor of shape (B,)."""
    _check_pair(sr, hr, "mse_y / psnr_y expect")
    sr = sr.contiguous().float()
    hr = hr.contiguous().float()
    B, _, H, W = sr.shape
    lib = _capi.load()
    scratch = torch.empty(int(lib.hitsir_psnr_y_scratch_doubles(B, H, W)), dtype=torch.float64, device=sr.device)
    out = torch.empty(B, dtype=torch.float64, device=sr.device)
    _call(lib.hitsir_psnr_y, sr.device, sr, hr, B, H, W, 1 if clip else 0, scratch, out)
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
    _check_pair(sr, hr, "ssim_y expects")
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
    scratch = torch.empty(int(lib.hitsir_ssim_y_scratch_doubles(B, H, W, g)), dtype=torch.float64, device=sr.device)
    out = torch.empty(B, dtype=torch.float64, device=sr.device)
    _call(lib.hitsir_ssim_y, sr.device, sr, hr, B, H, W, 1 if clip else 0, g, 1 if use_sample_covariance else 0, scratch, out)
    return out


def psnr_ssim_basicsr(sr_u8: torch.Tensor, hr_u8: torch.Tensor, crop_border: int, test_y_channel: bool = True):
    """BasicSR 1.4.2's `calculate_psnr` and `calculate_ssim` (basicsr/metrics/psnr_ssim.py), the scores of published SR tables, of
    every image of two uint8 (B,H,W,3) RGB CUDA batches, on the device (C ABI `hitsir_psnr_ssim_basicsr`).

    `crop_border` pixels are dropped on every side (BasicSR passes the scale factor); `test_y_channel` scores BasicSR's Y on the 0-255
    scale, else the three colour channels.  SSIM is the 11x11 Gaussian (sigma 1.5) window over the valid region, in float64.  Round an
    fp32 SR batch as BasicSR's `tensor2img` does first: ``to_uint8_hwc(sr, rounding="nearest")``.  Returns ``(psnr, ssim)``, float64
    (B,) CUDA tensors; psnr = 10 log10(255^2 / mse), +inf for identical images."""
    _check_pair(sr_u8, hr_u8, "psnr_ssim_basicsr expects", u8_hwc=True)
    c = int(crop_border)
    B, H, W, _ = sr_u8.shape
    if B == 0 or c < 0 or H - 2 * c < 11 or W - 2 * c < 11:
        raise ValueError(f"psnr_ssim_basicsr needs a non-empty batch, crop_border >= 0 and images of at least 11x11 after the crop, "
                         f"got {tuple(sr_u8.shape)} with crop_border={c}")
    sr_u8 = sr_u8.contiguous()
    hr_u8 = hr_u8.contiguous()
    y = 1 if test_y_channel else 0
    lib = _capi.load()
    scratch = torch.empty(int(lib.hitsir_basicsr_metrics_scratch_doubles(B, H, W, c, y)), dtype=torch.float64, device=sr_u8.device)
    mse = torch.empty(B, dtype=torch.float64, device=sr_u8.device)
    ssim = torch.empty(B, dtype=torch.float64, device=sr_u8.device)
    _call(lib.hitsir_psnr_ssim_basicsr, sr_u8.device, sr_u8, hr_u8, B, H, W, c, y, scratch, mse, ssim)
    return 10.0 * torch.log10(65025.0 / mse), ssim


def to_uint8_hwc(y: torch.Tensor, rounding: str = "truncate") -> torch.Tensor:
    """`to_pil_image(y.clip(0, 1))` of test_experiment.py:75-77 on the device: fp32 (B,C,H,W) -> uint8 (B,H,W,C), value * 255 truncated
    (C ABI `hitsir_f32nchw_to_u8hwc`).  The multi-GPU output gather moves this form: a quarter of the fp32 bytes.
    ``rounding="nearest"`` rounds half to even instead, as BasicSR's `tensor2img` does before its metrics (`hitsir_f32nchw_to_u8hwc_round`)."""
    if rounding not in ("truncate", "nearest"):
        raise ValueError(f"to_uint8_hwc: rounding must be 'truncate' or 'nearest', got {rounding!r}")
    if y.device.type != "cuda" or y.dim() != 4:
        raise RuntimeError("to_uint8_hwc expects a (B,C,H,W) CUDA tensor: there is no CPU path.")
    y = y.contiguous().float()
    B, C, H, W = y.shape
    out = torch.empty((B, H, W, C), dtype=torch.uint8, device=y.device)
    lib = _capi.load()
    _call(lib.hitsir_f32nchw_to_u8hwc if rounding == "truncate" else lib.hitsir_f32nchw_to_u8hwc_round, y.device, y, out, B, C, H, W)
    return out
