"""CPU oracle of the Y-channel SSIM (`hitsir_b200.ssim_y`) with an error bound derived from its arithmetic -- TEST INFRASTRUCTURE ONLY.

The reference evaluation (experiments/experiment.py:575-640) scores each image with
`skimage.metrics.structural_similarity(hr_y, sr_y, data_range=1)` on the Y planes of `oracle.metrics.y_channel` (`sr` clipped to
[0, 1] first).  requirements.txt pins scikit-image==0.24.0, which is neither vendored with the reference nor installed here, so:

* `ssim_y` restates skimage 0.24's `structural_similarity` for 2-D float32 images, line by line in numpy float32, with the
  `scipy.ndimage` calls it makes: `uniform_filter(size=7)` by default, `gaussian_filter(sigma=1.5, truncate=3.5, mode='reflect')` for
  `gaussian_weights=True`; `use_sample_covariance` picks cov_norm = win^2 / (win^2 - 1) (for the Gaussian window too) or 1; the
  result is `crop(S, pad).mean(dtype=float64)` with pad = (win - 1) // 2.
* `ssim_y_exact` is the same quantity in float64 from the same fp32 Y planes (products and window sums exact up to float64 rounding)
  together with a per-image bound on how far any evaluation with the arithmetic described at `ssim_y_exact` may lie from it: the
  float32 restatement above and the CUDA kernel both do.

SSIM parity with skimage itself is unpinned by a reference fixture (skimage is absent).  What pins the call is
`tests/test_ssim_oracle.py::test_reference_ssim_call_is_reproduced`: with the reference checkout at hand it reads every
`structural_similarity` call of experiments/experiment.py and checks that its arguments are ones `ssim_y` reproduces.
"""
from __future__ import annotations

import numpy as np
from scipy import ndimage

from oracle.metrics import y_channel

C1 = (0.01 * 1) ** 2          # (K1 * data_range) ** 2
C2 = (0.03 * 1) ** 2
SIGMA, TRUNCATE = 1.5, 3.5
U32 = 2.0 ** -24              # fp32 unit roundoff
F32 = np.float32


def win_size(gaussian_weights: bool) -> int:
    return 2 * int(TRUNCATE * SIGMA + 0.5) + 1 if gaussian_weights else 7


def _filter(a: np.ndarray, gaussian_weights: bool, origin: int = 0) -> np.ndarray:
    if gaussian_weights:
        g = ndimage.gaussian_filter(a, sigma=SIGMA, truncate=TRUNCATE, mode="reflect")
        # gaussian_filter takes no origin: a shifted window is the output moved by `origin` pixels along both axes (mutant only;
        # the wrapped rows and columns fall in the cropped border)
        return np.roll(g, origin, axis=(0, 1)) if origin else g
    return ndimage.uniform_filter(a, size=7, origin=origin)


def y_planes(sr, hr, clip: bool = True, channels=(0, 1, 2)):
    """fp32 Y planes (hr_y, sr_y), [N,H,W] each, as experiment.py forms them; `channels` reorders RGB (for a mutant only)."""
    sr = np.asarray(sr, dtype=np.float32)
    hr = np.asarray(hr, dtype=np.float32)
    if clip:
        sr = np.clip(sr, F32(0), F32(1))
    idx = list(channels)
    return y_channel(hr[:, idx]), y_channel(sr[:, idx])


def ssim_plane(im1: np.ndarray, im2: np.ndarray, gaussian_weights: bool = False, use_sample_covariance: bool = True,
               origin: int = 0, crop: bool = True, cov_norm_on: bool = True) -> float:
    """skimage 0.24 `structural_similarity(im1, im2, data_range=1, gaussian_weights=..., use_sample_covariance=...)` for 2-D float32
    images.  `origin`, `crop` and `cov_norm_on` exist only to build mutants (shifted window, no crop, cn dropped)."""
    im1 = np.asarray(im1, dtype=np.float32)
    im2 = np.asarray(im2, dtype=np.float32)
    ws = win_size(gaussian_weights)
    if min(im1.shape) < ws:
        raise ValueError("win_size exceeds image extent")
    NP = ws ** im1.ndim
    cov_norm = NP / (NP - 1) if use_sample_covariance else 1.0
    if not cov_norm_on:
        cov_norm = 1.0
    f = lambda a: _filter(a, gaussian_weights, origin)     # noqa: E731
    ux = f(im1)
    uy = f(im2)
    uxx = f(im1 * im1)
    uyy = f(im2 * im2)
    uxy = f(im1 * im2)
    # numpy: a Python float with a float32 array computes in float32
    vx = F32(cov_norm) * (uxx - ux * ux)
    vy = F32(cov_norm) * (uyy - uy * uy)
    vxy = F32(cov_norm) * (uxy - ux * uy)
    A1, A2, B1, B2 = (F32(2) * ux * uy + F32(C1), F32(2) * vxy + F32(C2), ux ** 2 + uy ** 2 + F32(C1), vx + vy + F32(C2))
    D = B1 * B2
    S = (A1 * A2) / D
    assert S.dtype == np.float32
    pad = (ws - 1) // 2
    if crop:
        S = S[pad:-pad, pad:-pad]
    return float(S.mean(dtype=np.float64))


def ssim_y(sr, hr, clip: bool = True, gaussian_weights: bool = False, use_sample_covariance: bool = True) -> np.ndarray:
    """Per-image SSIM of the Y channels, float64 [N]: structural_similarity(hr_y, sr_y, data_range=1) in float32 as skimage does."""
    x, y = y_planes(sr, hr, clip)
    return np.array([ssim_plane(x[i], y[i], gaussian_weights, use_sample_covariance) for i in range(x.shape[0])])


def _gamma(k: int) -> float:
    return k * U32 / (1 - k * U32)


def ssim_y_exact(sr, hr, clip: bool = True, gaussian_weights: bool = False, use_sample_covariance: bool = True):
    """(value, bound), float64 [N] each: the SSIM of the fp32 Y planes evaluated in float64, and a bound on |computed - value| for an
    evaluation that

    * forms the products x*x, y*y, x*y in fp32 (one rounding, relative u = 2^-24),
    * filters them with non-negative weights in float64 and rounds to fp32 at most twice: scipy rounds after each 1-D pass, the kernel
      sums the 2-D window in double and rounds once.  A moment m = sum w p therefore carries at most k = 3 fp32 roundings (second
      moments) or k = 2 (first moments): |computed - m| <= gamma_k * filter(|p|), which is gamma_k * m when the terms are
      non-negative, as they are for Y in [16/255, 235/255].  2^-44 * filter(|p|) covers the float64 sums and weights, and
      2^-40 * max|p| scipy's float64 running sum in `uniform_filter1d` (its error is relative to the largest window of the line);
    * then evaluates skimage's fp32 expression for S operation by operation, each operation rounded once (relative u).

    The bound is first order: each moment error and each rounding of an intermediate v (|delta v| <= u |v|) is carried to S by |dS/dv|
    at the exact values, S = A1 A2 / (B1 B2), plus the fp32 rounding of the constants cn, C1, C2.  Where a moment enters S along several
    paths (ux in A1, B1, A2 and B2) its derivative is taken as a whole, so the near-cancellation of those paths when sr ~ hr is not
    counted twice.  A second-order remainder 16 r^2 |S| is added, with r the largest relative error of A1, A2, B1, B2 from a plain
    interval propagation of the same errors.  The image bound is the mean of the per-pixel bounds over the cropped interior plus the
    float64 summation of the mean."""
    x32, y32 = y_planes(sr, hr, clip)
    ws = win_size(gaussian_weights)
    NP = ws * ws
    cn = NP / (NP - 1) if use_sample_covariance else 1.0
    e_cn = abs(float(F32(cn)) - cn)
    e_c1 = abs(float(F32(C1)) - C1)
    e_c2 = abs(float(F32(C2)) - C2)
    u = U32
    pad = (ws - 1) // 2
    g1, g2 = _gamma(2) + 2.0 ** -44, _gamma(3) + 2.0 ** -44
    values, bounds = [], []
    for i in range(x32.shape[0]):
        x = x32[i].astype(np.float64)
        y = y32[i].astype(np.float64)
        f = lambda a: _filter(a, gaussian_weights)[pad:-pad, pad:-pad]     # noqa: E731
        ux, uy, uxx, uyy, uxy = f(x), f(y), f(x * x), f(y * y), f(x * y)
        slack1 = 2.0 ** -40 * max(np.abs(x).max(), np.abs(y).max())
        slack2 = 2.0 ** -40 * max((x * x).max(), (y * y).max(), np.abs(x * y).max())
        ex, ey = g1 * f(np.abs(x)) + slack1, g1 * f(np.abs(y)) + slack1
        exx, eyy, exy = g2 * uxx + slack2, g2 * uyy + slack2, g2 * f(np.abs(x * y)) + slack2

        d1, d2, d3 = uxx - ux * ux, uyy - uy * uy, uxy - ux * uy
        vx, vy, vxy = cn * d1, cn * d2, cn * d3
        t1 = 2.0 * ux * uy
        A1, A2 = t1 + C1, 2.0 * vxy + C2
        s1 = ux * ux + uy * uy
        B1 = s1 + C1
        s2 = vx + vy
        B2 = s2 + C2
        S = (A1 * A2) / (B1 * B2)
        aS = np.abs(S)
        kA1, kA2, kB1, kB2 = aS / np.abs(A1), aS / np.abs(A2), aS / B1, aS / B2      # |dS/dA1| ...
        # moments
        lin = (cn * kB2 * (exx + eyy) + 2 * cn * kA2 * exy
               + np.abs(S * (2 * uy / A1 - 2 * ux / B1 - 2 * cn * uy / A2 + 2 * cn * ux / B2)) * ex
               + np.abs(S * (2 * ux / A1 - 2 * uy / B1 - 2 * cn * ux / A2 + 2 * cn * uy / B2)) * ey)
        # constants
        lin += np.abs(S * (2 * d3 / A2 - (d1 + d2) / B2)) * e_cn + np.abs(S * (1 / A1 - 1 / B1)) * e_c1 + np.abs(S * (1 / A2 - 1 / B2)) * e_c2
        # one rounding per operation: products ux*ux, uy*uy, ux*uy; differences; * cn; A1, A2, B1, B2 and their parts; N, D, S
        lin += u * (cn * kB2 * (ux * ux + uy * uy + np.abs(d1) + np.abs(d2)) + kB2 * (np.abs(vx) + np.abs(vy) + np.abs(s2))
                    + 2 * cn * kA2 * (np.abs(ux * uy) + np.abs(d3)) + 2 * kA2 * np.abs(vxy)
                    + kA1 * np.abs(t1) + kB1 * (ux * ux + uy * uy + s1)
                    + kA1 * np.abs(A1) + kA2 * np.abs(A2) + kB1 * B1 + kB2 * B2 + 3 * aS)
        # second-order remainder from a plain interval propagation of the same errors
        e_var = lambda m, em, a, ea, b, eb: cn * (em + np.abs(a) * eb + np.abs(b) * ea + ea * eb) + 4 * u * np.abs(m)   # noqa: E731
        evx, evy, evxy = e_var(uxx, exx, ux, ex, ux, ex), e_var(uyy, eyy, uy, ey, uy, ey), e_var(uxy, exy, ux, ex, uy, ey)
        r = np.maximum.reduce([(2 * np.abs(ux) * ey + 2 * np.abs(uy) * ex + 2 * ex * ey + e_c1) / np.abs(A1) + 3 * u,
                               (2 * evxy + e_c2) / np.abs(A2) + 2 * u,
                               (2 * np.abs(ux) * ex + 2 * np.abs(uy) * ey + ex * ex + ey * ey + e_c1) / B1 + 3 * u,
                               (evx + evy + e_c2) / B2 + 2 * u])
        eS = lin + 16 * r * r * aS + 2.0 ** -40                 # + the float64 evaluation of S itself
        eS = np.where(r < 0.25, eS, np.inf)
        n = S.size
        values.append(S.mean())
        bounds.append(eS.mean() + 2 * n * 2.0 ** -53 * (aS.mean() + eS.mean()))
    return np.array(values), np.array(bounds)


def ssim_direct(x: np.ndarray, y: np.ndarray, gaussian_weights: bool, use_sample_covariance: bool) -> float:
    """float64 SSIM of two small 2-D planes by explicit window sums, no scipy: an independent check of the window's centring, its
    weights and the crop."""
    import math
    ws = win_size(gaussian_weights)
    p = (ws - 1) // 2
    if gaussian_weights:
        w1 = [math.exp(-0.5 * (j - p) ** 2 / SIGMA ** 2) for j in range(ws)]
        w1 = [w / sum(w1) for w in w1]
    else:
        w1 = [1.0 / ws] * ws
    cn = ws * ws / (ws * ws - 1) if use_sample_covariance else 1.0
    H, W = x.shape
    total, count = 0.0, 0
    for i in range(p, H - p):
        for j in range(p, W - p):
            m = [0.0] * 5
            for a in range(ws):
                for b in range(ws):
                    w = w1[a] * w1[b]
                    xv, yv = float(x[i - p + a, j - p + b]), float(y[i - p + a, j - p + b])
                    for q, v in enumerate((xv, yv, xv * xv, yv * yv, xv * yv)):
                        m[q] += w * v
            ux, uy, uxx, uyy, uxy = m
            vx, vy, vxy = cn * (uxx - ux * ux), cn * (uyy - uy * uy), cn * (uxy - ux * uy)
            total += ((2 * ux * uy + C1) * (2 * vxy + C2)) / ((ux * ux + uy * uy + C1) * (vx + vy + C2))
            count += 1
    return total / count


def inputs(kind: str, B: int, H: int, W: int, seed: int):
    """Seeded (sr, hr) fp32 [B,3,H,W] pairs: 'random' (uniform hr), 'smooth' (low-frequency hr) and 'flat1' (hr with a flat region
    near Y = 1, where the window variances vanish and `sr`'s clip matters); `sr` = hr + N(0, 0.03), so it leaves [0, 1]."""
    rng = np.random.Generator(np.random.PCG64(seed))
    if kind == "random":
        hr = rng.random((B, 3, H, W), dtype=np.float32)
    else:
        yy, xx = np.meshgrid(np.arange(H, dtype=np.float64), np.arange(W, dtype=np.float64), indexing="ij")
        hr = np.empty((B, 3, H, W), np.float32)
        for b in range(B):
            for c in range(3):
                # periods of 48 to 128 pixels: smooth at the scale of the window whatever the image size
                fy, fx, ph = rng.uniform(1 / 128, 1 / 48), rng.uniform(1 / 128, 1 / 48), rng.uniform(0, 2 * np.pi)
                hr[b, c] = 0.5 + 0.35 * np.sin(2 * np.pi * (fy * yy + fx * xx) + ph)
        if kind == "flat1":
            # the left quarter is flat near 1 (tiny texture), the rest smooth
            hr[:, :, :, : max(1, W // 4)] = 0.985 + 0.01 * rng.random((B, 3, H, max(1, W // 4)), dtype=np.float32)
        elif kind != "smooth":
            raise ValueError(kind)
    sr = (hr + rng.normal(0.0, 0.03, hr.shape).astype(np.float32)).astype(np.float32)
    return sr, hr
