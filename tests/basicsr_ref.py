"""CPU oracle of BasicSR's PSNR / SSIM (`hitsir_b200.psnr_ssim_basicsr`) with an error bound derived from its arithmetic -- TEST
INFRASTRUCTURE ONLY.

Published SR tables are scored by BasicSR 1.4.2's `calculate_psnr` / `calculate_ssim` (basicsr/metrics/psnr_ssim.py, with
`to_y_channel` of metric_util.py and `bgr2ycbcr` of utils/color_util.py) on the uint8 images `tensor2img` makes.  BasicSR holds images
in BGR.  This module restates, with numpy and cv2:

* `tensor2img`, `to_y_channel`, `calculate_psnr`, `calculate_ssim` line by line (BGR HWC uint8 in, as BasicSR takes them);
  `psnr_ssim` applies them to RGB batches (B,H,W,3).  These are what the device is judged against for parity, and
  `tests/test_basicsr_oracle.py` checks them bitwise against the vendored BasicSR when a reference checkout is at hand;
* `y_device_order`: the Y formula in the IEEE operation order of `y_basicsr` (ycbcr.cuh);
* `psnr_ssim_exact`: the same scores in extended precision (`np.longdouble` separable window sums) with a per-image bound on how far
  an fp64 evaluation by direct window sums may lie from them (the CUDA kernel is one), and optionally cv2's DFT-based `filter2D`.
"""
from __future__ import annotations

import importlib.util
import os
import sys
import types

import cv2
import numpy as np

KERNEL = cv2.getGaussianKernel(11, 1.5)[:, 0]          # float64 (11,), BasicSR's window is outer(KERNEL, KERNEL)
C1 = (0.01 * 255) ** 2
C2 = (0.03 * 255) ** 2
U = 2.0 ** -53                                         # fp64 unit roundoff
UL = float(np.finfo(np.longdouble).eps) / 2            # unit roundoff of the extended-precision reference
# cv2.filter2D on float64 with an 11x11 kernel goes through OpenCV's DFT, whose error is relative to the largest value of the plane
# rather than to each window: up to ~1.7e-13 on 0-255 data (about 6 u * 255).  DFT_ALLOWANCE * max|p| per moment covers that 85x over.
DFT_ALLOWANCE = 2.0 ** -44


# ---- BasicSR, restated ---------------------------------------------------------------------------------------------------------------

def tensor2img(x: np.ndarray) -> np.ndarray:
    """basicsr/utils/img_util.py tensor2img of an fp32 (B,C,H,W) batch in [0, 1] (min_max=(0, 1), out_type=uint8), kept RGB and
    batched: (B,H,W,C) uint8.  `(x - 0) / (1 - 0)` is the identity on fp32 and is left out."""
    x = np.clip(np.asarray(x, dtype=np.float32), 0, 1)
    v = (x * 255.0).round()                            # float32 array * Python float stays float32; round half to even
    assert v.dtype == np.float32
    return v.astype(np.uint8).transpose(0, 2, 3, 1).copy()


def to_y_channel(img: np.ndarray) -> np.ndarray:
    """metric_util.to_y_channel of a BGR uint8 HWC image: float32 (H,W,1) on the 0-255 scale."""
    img = img.astype(np.float32) / 255.
    out = np.dot(img, [24.966, 128.553, 65.481]) + 16.0      # bgr2ycbcr(y_only=True), float64
    out = (out / 255.).astype(np.float32)                   # _convert_output_type_range to float32
    return out[..., None] * 255.


def _crop(img, c):
    return img[c:-c, c:-c, ...] if c != 0 else img


def calculate_psnr(img, img2, crop_border, test_y_channel=False):
    assert img.shape == img2.shape
    img, img2 = _crop(img, crop_border), _crop(img2, crop_border)
    if test_y_channel:
        img, img2 = to_y_channel(img), to_y_channel(img2)
    img = img.astype(np.float64)
    img2 = img2.astype(np.float64)
    mse = np.mean((img - img2) ** 2)
    if mse == 0:
        return float("inf")
    return 10. * np.log10(255. * 255. / mse)


def mse_basicsr(img, img2, crop_border, test_y_channel=False):
    """The `mse` that calculate_psnr forms."""
    img, img2 = _crop(img, crop_border), _crop(img2, crop_border)
    if test_y_channel:
        img, img2 = to_y_channel(img), to_y_channel(img2)
    return np.mean((img.astype(np.float64) - img2.astype(np.float64)) ** 2)


def _ssim(img, img2, window=None, cn=1.0, valid=True, c1=C1, c2=C2):
    """psnr_ssim._ssim; `window`, `cn`, `valid` and `c1`/`c2` other than their defaults exist only to build mutants."""
    if window is None:
        window = np.outer(KERNEL, KERNEL.transpose())
    r = window.shape[0] // 2
    crop = (lambda a: a[r:-r, r:-r]) if valid else (lambda a: a)      # noqa: E731
    mu1 = crop(cv2.filter2D(img, -1, window))
    mu2 = crop(cv2.filter2D(img2, -1, window))
    mu1_sq = mu1 ** 2
    mu2_sq = mu2 ** 2
    mu1_mu2 = mu1 * mu2
    sigma1_sq = cn * (crop(cv2.filter2D(img ** 2, -1, window)) - mu1_sq)
    sigma2_sq = cn * (crop(cv2.filter2D(img2 ** 2, -1, window)) - mu2_sq)
    sigma12 = cn * (crop(cv2.filter2D(img * img2, -1, window)) - mu1_mu2)
    ssim_map = ((2 * mu1_mu2 + c1) * (2 * sigma12 + c2)) / ((mu1_sq + mu2_sq + c1) * (sigma1_sq + sigma2_sq + c2))
    return ssim_map.mean()


def calculate_ssim(img, img2, crop_border, test_y_channel=False, **mutant):
    assert img.shape == img2.shape
    img, img2 = _crop(img, crop_border), _crop(img2, crop_border)
    if test_y_channel:
        img, img2 = to_y_channel(img), to_y_channel(img2)
    img = img.astype(np.float64)
    img2 = img2.astype(np.float64)
    ssims = [_ssim(img[..., i], img2[..., i], **mutant) for i in range(img.shape[2])]
    return np.array(ssims).mean()


def bgr(x_rgb: np.ndarray) -> np.ndarray:
    return np.ascontiguousarray(x_rgb[..., ::-1])


def psnr_ssim(sr_u8, hr_u8, crop_border, test_y_channel=True):
    """BasicSR's (psnr, ssim) of every image of two RGB uint8 (B,H,W,3) batches, float64 (B,) each; SR is BasicSR's `img`."""
    p = [calculate_psnr(bgr(s), bgr(h), crop_border, test_y_channel) for s, h in zip(sr_u8, hr_u8)]
    s = [calculate_ssim(bgr(s), bgr(h), crop_border, test_y_channel) for s, h in zip(sr_u8, hr_u8)]
    return np.array(p, np.float64), np.array(s, np.float64)


def y_device_order(r, g, b) -> np.ndarray:
    """y_basicsr of ycbcr.cuh on uint8 arrays, operation by operation (numpy's elementwise float64 ops do not contract)."""
    f = lambda v: (np.asarray(v).astype(np.float32) / np.float32(255)).astype(np.float64)     # noqa: E731
    y = ((24.966 * f(b) + 128.553 * f(g)) + 65.481 * f(r)) + 16.0
    return (y / 255.0).astype(np.float32) * np.float32(255)


# ---- extended-precision reference and bound ------------------------------------------------------------------------------------------

def _valid_filter(p, k):
    """Separable correlation with outer(k, k) over the 'valid' region, in p's dtype."""
    H, W = p.shape
    n = len(k)
    h = sum(k[t] * p[:, t:W - n + 1 + t] for t in range(n))
    return sum(k[t] * h[t:H - n + 1 + t, :] for t in range(n))


def _gamma(k: int, u: float = U) -> float:
    return k * u / (1 - k * u)


def _sum_depth(n: int) -> int:
    # depth of any fixed-order summation of n values that the bound covers: the kernel's thread -> warp -> CTA -> tile order
    # (< 30 + n / 32768) and numpy's pairwise sum (< 16 + log2 n) both stay below it
    return 64 + n // 1024


def ssim_plane_exact(a: np.ndarray, b: np.ndarray, dft: bool = False):
    """(value, bound) for one plane pair (float64 values, cropped): BasicSR's _ssim with the window sums and S in np.longdouble, and a
    bound on |computed - value| for an evaluation that

    * forms the products a*a, b*b, a*b in float64 (exact: the planes are fp32 Y values or integers),
    * sums each window with weights outer(k, k) in float64, separably (11 + 11 terms) or with the 121 weights rounded once: a moment
      m = sum W p of non-negative terms (every plane value is >= 0) carries at most gamma_23 * m; with `dft`, cv2.filter2D's DFT,
      DFT_ALLOWANCE * max|p| more,
    * evaluates BasicSR's expression for S in float64 operation by operation, each operation rounded once (relative u = 2^-53),
    * and sums the map in a fixed order of depth at most _sum_depth(n), then divides by n.

    As in tests/ssim_ref.py the bound is first order: each moment error and each rounding of an intermediate is carried to S by |dS/dv|
    at the exact values (a moment entering S along several paths by its whole derivative), plus a second-order remainder 16 r^2 |S|
    with r the largest relative error of the four factors from a plain interval propagation.  The reference's own extended-precision
    error is the same expression scaled by UL / U and is added."""
    L = np.longdouble
    k = KERNEL.astype(L)
    A, B = a.astype(L), b.astype(L)
    mu1, mu2, e11, e22, e12 = (_valid_filter(p, k) for p in (A, B, A * A, B * B, A * B))
    m1s, m2s, m12 = mu1 * mu1, mu2 * mu2, mu1 * mu2
    s1, s2, s12 = e11 - m1s, e22 - m2s, e12 - m12
    A1, A2 = 2 * m12 + L(C1), 2 * s12 + L(C2)
    B1, B2 = m1s + m2s + L(C1), s1 + s2 + L(C2)
    S = (A1 * A2) / (B1 * B2)

    f64 = lambda v: np.asarray(v, dtype=np.float64)     # noqa: E731
    mu1, mu2, e11, e22, e12, m1s, m2s, m12, s1, s2, s12, A1, A2, B1, B2 = map(f64, (mu1, mu2, e11, e22, e12, m1s, m2s, m12, s1, s2, s12,
                                                                                  A1, A2, B1, B2))
    Sd = f64(S)
    aS = np.abs(Sd)
    g = _gamma(23)
    slack1 = DFT_ALLOWANCE * max(np.abs(a).max(), np.abs(b).max()) if dft else 0.0
    slack2 = DFT_ALLOWANCE * max((a * a).max(), (b * b).max()) if dft else 0.0
    em1, em2 = g * mu1 + slack1, g * mu2 + slack1
    e_11, e_22, e_12 = g * e11 + slack2, g * e22 + slack2, g * e12 + slack2
    kA1, kA2, kB1, kB2 = aS / np.abs(A1), aS / np.abs(A2), aS / B1, aS / B2
    lin = (kB2 * (e_11 + e_22) + 2 * kA2 * e_12
           + np.abs(Sd * (2 * mu2 / A1 - 2 * mu2 / A2 - 2 * mu1 / B1 + 2 * mu1 / B2)) * em1
           + np.abs(Sd * (2 * mu1 / A1 - 2 * mu1 / A2 - 2 * mu2 / B1 + 2 * mu2 / B2)) * em2)
    # one rounding per operation: mu1^2, mu2^2 (into B1 and B2), mu1 mu2 (into A1 and A2), the three differences, the sums, + c1 / c2,
    # the two products and the division
    lin += U * ((kB1 + kB2) * (m1s + m2s) + 2 * (kA1 + kA2) * np.abs(m12) + 2 * kA2 * np.abs(s12) + kB2 * (np.abs(s1) + np.abs(s2))
                + kB1 * (m1s + m2s) + kB2 * np.abs(s1 + s2) + kA1 * np.abs(A1) + kA2 * np.abs(A2) + kB1 * B1 + kB2 * B2 + 3 * aS)
    e_var = lambda m, em, x, ex, y, ey: em + np.abs(x) * ey + np.abs(y) * ex + ex * ey + 4 * U * np.abs(m)    # noqa: E731
    es1, es2, es12 = e_var(e11, e_11, mu1, em1, mu1, em1), e_var(e22, e_22, mu2, em2, mu2, em2), e_var(e12, e_12, mu1, em1, mu2, em2)
    r = np.maximum.reduce([(2 * np.abs(mu1) * em2 + 2 * np.abs(mu2) * em1 + 2 * em1 * em2) / np.abs(A1) + 3 * U,
                           2 * es12 / np.abs(A2) + 2 * U,
                           (2 * np.abs(mu1) * em1 + 2 * np.abs(mu2) * em2 + em1 * em1 + em2 * em2) / B1 + 3 * U,
                           (es1 + es2) / B2 + 2 * U])
    eS = (lin + 16 * r * r * aS) * (1 + UL / U)
    eS = np.where(r < 0.25, eS, np.inf)
    n = S.size
    value = float(S.mean())
    bound = float(eS.mean()) + (_gamma(_sum_depth(n)) + U) * (float(aS.mean()) + float(eS.mean())) + UL * n * float(aS.mean())
    return value, bound


def _planes(img_rgb_u8, c, test_y_channel):
    """float64 planes (P,Hc,Wc) of one RGB uint8 image after the crop, in BasicSR's channel order (BGR when not Y)."""
    img = _crop(bgr(img_rgb_u8), c)
    v = to_y_channel(img) if test_y_channel else img
    return np.moveaxis(v.astype(np.float64), 2, 0)


def psnr_ssim_exact(sr_u8, hr_u8, crop_border, test_y_channel=True, dft=False):
    """Per image (mse, mse_bound, ssim, ssim_bound), float64 (B,) each.  mse: sum of squared differences in np.longdouble over the crop
    (RGB: exact integers, bound 0; Y: each square rounded once and summed in a fixed order of depth _sum_depth(n)).  ssim: the planes'
    ssim_plane_exact, averaged over the planes in BasicSR's order ((B + G) + R) / 3 (three more roundings)."""
    out = []
    for s, h in zip(sr_u8, hr_u8):
        a, b = _planes(s, crop_border, test_y_channel), _planes(h, crop_border, test_y_channel)
        d = a.astype(np.longdouble) - b.astype(np.longdouble)
        sq = d * d
        n = sq.size
        mse = float(sq.sum() / n)
        mse_bound = 0.0 if not test_y_channel else (U + _gamma(_sum_depth(n)) + U) * mse * (1 + UL / U) + UL * n * mse
        vb = [ssim_plane_exact(a[p], b[p], dft) for p in range(a.shape[0])]
        val = sum(v for v, _ in vb) / len(vb)
        bnd = sum(e for _, e in vb) / len(vb) + (4 * U * (abs(val) + 1) if len(vb) > 1 else 0.0)
        out.append((mse, mse_bound, val, bnd))
    return tuple(np.array(col, np.float64) for col in zip(*out))


# ---- inputs ----------------------------------------------------------------------------------------------------------------------------

def inputs(kind: str, B: int, H: int, W: int, seed: int):
    """Seeded (sr_f32, hr_u8): hr_u8 uint8 (B,H,W,3), sr_f32 fp32 (B,3,H,W) = hr / 255 + noise, which leaves [0, 1] and is rounded by
    tensor2img.  'random' (uniform hr), 'smooth' (low-frequency hr), 'flat0' / 'flat255' (hr flat within 3 levels of 0 or 255)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    if kind == "random":
        hr = rng.integers(0, 256, (B, H, W, 3), dtype=np.uint8)
    elif kind == "smooth":
        yy, xx = np.meshgrid(np.arange(H, dtype=np.float64), np.arange(W, dtype=np.float64), indexing="ij")
        hr = np.empty((B, H, W, 3), np.uint8)
        for b in range(B):
            for c in range(3):
                fy, fx, ph = rng.uniform(1 / 128, 1 / 48), rng.uniform(1 / 128, 1 / 48), rng.uniform(0, 2 * np.pi)
                hr[b, :, :, c] = np.round(127.5 + 90 * np.sin(2 * np.pi * (fy * yy + fx * xx) + ph)).astype(np.uint8)
    elif kind in ("flat0", "flat255"):
        t = rng.integers(0, 3, (B, H, W, 3))
        hr = (t if kind == "flat0" else 255 - t).astype(np.uint8)
    else:
        raise ValueError(kind)
    noise = 0.004 if kind.startswith("flat") else 0.03
    sr = (hr.transpose(0, 3, 1, 2).astype(np.float32) / np.float32(255) + rng.normal(0.0, noise, (B, 3, H, W))).astype(np.float32)
    return sr, hr


# ---- the vendored BasicSR ----------------------------------------------------------------------------------------------------------

def load_vendored(root: str):
    """basicsr.metrics.psnr_ssim of the reference checkout's BasicSR_master, loaded with its two helper modules without executing
    basicsr/__init__ (which imports the whole training stack): the parent packages and the registry are stubs, and sys.modules is
    restored afterwards."""
    base = os.path.join(root, "BasicSR_master", "basicsr")
    names = ["basicsr", "basicsr.utils", "basicsr.metrics", "basicsr.utils.registry", "basicsr.utils.color_util",
             "basicsr.metrics.metric_util", "basicsr.metrics.psnr_ssim"]
    saved = {n: sys.modules.get(n) for n in names}

    class _Registry:
        def register(self, obj=None):
            return (lambda f: f) if obj is None else obj

    def _load(name, rel):
        spec = importlib.util.spec_from_file_location(name, os.path.join(base, rel))
        mod = importlib.util.module_from_spec(spec)
        sys.modules[name] = mod
        spec.loader.exec_module(mod)
        return mod

    try:
        for n in names[:3]:
            sys.modules[n] = types.ModuleType(n)
            sys.modules[n].__path__ = []
        reg = types.ModuleType("basicsr.utils.registry")
        reg.METRIC_REGISTRY = _Registry()
        sys.modules["basicsr.utils.registry"] = reg
        color = _load("basicsr.utils.color_util", os.path.join("utils", "color_util.py"))
        sys.modules["basicsr.utils"].bgr2ycbcr = color.bgr2ycbcr
        _load("basicsr.metrics.metric_util", os.path.join("metrics", "metric_util.py"))
        return _load("basicsr.metrics.psnr_ssim", os.path.join("metrics", "psnr_ssim.py"))
    finally:
        for n, m in saved.items():
            if m is None:
                sys.modules.pop(n, None)
            else:
                sys.modules[n] = m


def vendored_path(root: str) -> str:
    return os.path.join(root, "BasicSR_master", "basicsr", "metrics", "psnr_ssim.py")


def gaussian_formula() -> np.ndarray:
    """exp(-x^2 / (2 sigma^2)) normalised, x = -5..5, sigma = 1.5: the textbook form of cv2.getGaussianKernel(11, 1.5)."""
    x = np.arange(-5, 6, dtype=np.float64)
    e = np.exp(-x * x / (2 * 1.5 * 1.5))
    return e / e.sum()

