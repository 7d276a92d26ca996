"""CPU restatements of the two bicubic resizers (`hitsir_b200.resize_bicubic`) with an error bound for the fp32 one -- TEST
INFRASTRUCTURE ONLY.

* `pil_resize`: Pillow 12.2's ``Image.resize(size, Image.BICUBIC)`` for modes L / RGB (libImaging/Resample.c: precompute_coeffs,
  normalize_coeffs_8bpc, ImagingResampleHorizontal_8bpc / Vertical_8bpc), tap tables in Python floats operation by operation as the C
  code writes them, the passes in integers.  `tests/test_resize_oracle.py` checks it against Pillow bit for bit; the CUDA kernel
  builds the same tables with explicitly rounded double operations, so the GPU test compares it against Pillow directly.
* `matlab_resize`: MATLAB ``imresize(x, scale, 'bicubic')`` as BasicSR's ``calculate_weights_indices`` + ``imresize`` compute it,
  in float64 (weights and sums), H pass then W pass.
* `matlab_bound`: per-pixel bound on |computed - matlab_resize| for an evaluation with fp32-rounded weights and fp32 FMA sums in tap
  order, as the CUDA kernel does.

Keyword arguments that change the arithmetic (`a`, `precision_bits`, `vertical_first`, `antialias`, `boundary`) exist to build
mutants.
"""
from __future__ import annotations

import math

import numpy as np

U32 = 2.0 ** -24          # fp32 unit roundoff


# ---- Pillow -------------------------------------------------------------------------------------------------------------------------
def pil_filter(x: float, a: float = -0.5) -> float:
    if x < 0.0:
        x = -x
    if x < 1.0:
        return ((a + 2.0) * x - (a + 3.0)) * x * x + 1
    if x < 2.0:
        return (((x - 5) * x + 8) * x - 4) * a
    return 0.0


def pil_coeffs(in_size: int, out_size: int, a: float = -0.5, precision_bits: int = 22):
    """[(xmin, [fixed-point coefficients])] per output index: precompute_coeffs + normalize_coeffs_8bpc with box = (0, in_size)."""
    scale = float(in_size) / out_size
    filterscale = max(scale, 1.0)
    support = 2.0 * filterscale
    table = []
    for xx in range(out_size):
        center = 0.0 + (xx + 0.5) * scale
        ss = 1.0 / filterscale
        xmin = max(int(center - support + 0.5), 0)
        xmax = min(int(center + support + 0.5), in_size) - xmin
        k = [pil_filter((x + xmin - center + 0.5) * ss, a) for x in range(xmax)]
        ww = 0.0
        for w in k:
            ww += w
        if ww != 0.0:
            k = [w / ww for w in k]
        one = float(1 << precision_bits)
        table.append((xmin, [int(-0.5 + w * one) if w < 0 else int(0.5 + w * one) for w in k]))
    return table


def _pil_pass(img: np.ndarray, axis: int, out_size: int, a: float, precision_bits: int) -> np.ndarray:
    """One 8bpc pass along `axis` (0 = rows / vertical, 1 = columns / horizontal) of an int64 [H, W, C] image."""
    table = pil_coeffs(img.shape[axis], out_size, a, precision_bits)
    m = np.zeros((out_size, img.shape[axis]), np.int64)
    for o, (xmin, k) in enumerate(table):
        m[o, xmin:xmin + len(k)] = k
    acc = np.einsum("oi,hic->hoc", m, img) if axis == 1 else np.einsum("oi,iwc->owc", m, img)
    acc = acc + (1 << (precision_bits - 1))
    return np.clip(acc >> precision_bits, 0, 255)


def pil_resize(img: np.ndarray, out_h: int, out_w: int, a: float = -0.5, precision_bits: int = 22,
               vertical_first: bool = False) -> np.ndarray:
    """uint8 [H, W] or [H, W, C] -> uint8 [out_h, out_w(, C)]: Image.resize((out_w, out_h), Image.BICUBIC).  Horizontal pass
    first (each skipped when its axis keeps its size), uint8 between the passes; Pillow's restriction of the horizontal pass to the
    rows the vertical pass reads changes no value and is left out."""
    x = np.asarray(img)
    squeeze = x.ndim == 2
    x = (x[:, :, None] if squeeze else x).astype(np.int64)
    passes = [(1, out_w), (0, out_h)]
    for axis, n in (passes[::-1] if vertical_first else passes):
        if x.shape[axis] != n:
            x = _pil_pass(x, axis, n, a, precision_bits)
    x = x.astype(np.uint8)
    return x[:, :, 0] if squeeze else x


# ---- MATLAB / BasicSR ---------------------------------------------------------------------------------------------------------------
def matlab_cubic(x: float, a: float = -0.5) -> float:
    """BasicSR's cubic for a = -0.5: (1.5|x|^3 - 2.5|x|^2 + 1) on |x| <= 1, (-0.5|x|^3 + 2.5|x|^2 - 4|x| + 2) on (1, 2]; the
    general Keys form for another `a` (mutant only)."""
    ax = abs(x)
    a2 = ax * ax
    a3 = a2 * ax
    if ax <= 1.0:
        return (a + 2.0) * a3 - (a + 3.0) * a2 + 1.0
    if ax <= 2.0:
        return a * a3 - 5.0 * a * a2 + 8.0 * a * ax - 4.0 * a
    return 0.0


def matlab_out_size(in_size: int, scale: float) -> int:
    return math.ceil(in_size * scale)


def matlab_weights(in_size: int, scale: float, a: float = -0.5, antialias: bool = True, drop_zero_columns: bool = True):
    """(weights, indices), float64 / int64 [out, taps]: calculate_weights_indices(in, ceil(in*scale), scale, 'cubic', 4, antialias)
    in float64 with 0-based input indices before the boundary is applied.  MATLAB drops an all-zero first / last tap column."""
    out = matlab_out_size(in_size, scale)
    aa = scale < 1.0 and antialias
    width = 4.0 / scale if aa else 4.0
    p = math.ceil(width) + 2
    w = np.zeros((out, p))
    idx = np.zeros((out, p), np.int64)
    for o in range(out):
        u = (o + 1) / scale + 0.5 * (1.0 - 1.0 / scale)
        left = math.floor(u - width * 0.5)
        row = []
        for k in range(p):
            d = u - (left + k)
            row.append(scale * matlab_cubic(d * scale, a) if aa else matlab_cubic(d, a))
        s = 0.0
        for v in row:
            s += v
        w[o] = [v / s for v in row]
        idx[o] = np.arange(left - 1, left - 1 + p)
    if drop_zero_columns:
        lo = 1 if not np.any(w[:, 0]) else 0
        hi = p - 1 if not np.any(w[:, -1]) else p
        w, idx = w[:, lo:hi], idx[:, lo:hi]
    return w, idx


def mirror(i: np.ndarray, n: int) -> np.ndarray:
    """Half-sample symmetric boundary: -1 -> 0, -2 -> 1, n -> n-1 (BasicSR pads with the flipped edge rows)."""
    i = np.mod(i, 2 * n)
    return np.where(i < n, i, 2 * n - 1 - i)


def matlab_matrix(in_size: int, scale: float, absolute: bool = False, boundary: str = "mirror", **kw) -> np.ndarray:
    """Dense [out, in] float64 resampling matrix of one axis (|weights| summed per input index when `absolute`)."""
    w, idx = matlab_weights(in_size, scale, **kw)
    j = mirror(idx, in_size) if boundary == "mirror" else np.clip(idx, 0, in_size - 1)
    m = np.zeros((w.shape[0], in_size))
    np.add.at(m, (np.repeat(np.arange(w.shape[0]), w.shape[1]), j.ravel()), (np.abs(w) if absolute else w).ravel())
    return m


def matlab_resize(x: np.ndarray, scale: float, boundary: str = "mirror", **kw) -> np.ndarray:
    """float64 [..., H, W] -> [..., ceil(H*scale), ceil(W*scale)]: the H pass, then the W pass."""
    x = np.asarray(x, dtype=np.float64)
    mh = matlab_matrix(x.shape[-2], scale, boundary=boundary, **kw)
    mw = matlab_matrix(x.shape[-1], scale, boundary=boundary, **kw)
    return np.einsum("oh,...hw->...ow", mh, x) @ mw.T


def _gamma(k: int) -> float:
    return k * U32 / (1 - k * U32)


def matlab_bound(x: np.ndarray, scale: float) -> np.ndarray:
    """Per-pixel bound on |computed - matlab_resize(x, scale)| for a separable evaluation, in either pass order, that

    * rounds each float64 weight to fp32 once (relative u = 2^-24), and
    * sums the p taps of an output (p = ceil(width) + 2, zero taps included) in fp32, each step an FMA or a rounded product and sum.

    A pass over values v with weights w then errs by at most e(v) = (u + gamma_{2p} (1 + u)) sum_k |w_k| |v_k| from its exact
    result, and the second pass carries the first pass's error e1 through sum |w| e1.  With |M| the matrices of summed |weights|:
    bound = |M_2| e1 + c |M_2| (|M_1| |x| + e1), e1 = c |M_1| |x|, c = u + gamma_2p (1 + u); the larger of the two orders is taken,
    plus 2^-45 |M_2| |M_1| |x| for the float64 reference itself."""
    x = np.abs(np.asarray(x, dtype=np.float64))
    p = matlab_weights(x.shape[-2] if x.shape[-2] > 0 else 1, scale, drop_zero_columns=False)[0].shape[1]
    c = U32 + _gamma(2 * p) * (1 + U32)
    ah = matlab_matrix(x.shape[-2], scale, absolute=True)
    aw = matlab_matrix(x.shape[-1], scale, absolute=True)
    along_h = lambda v: np.einsum("oh,...hw->...ow", ah, v)     # noqa: E731
    along_w = lambda v: v @ aw.T                                # noqa: E731
    bounds = []
    for first, second in ((along_h, along_w), (along_w, along_h)):
        a1 = first(x)
        e1 = c * a1
        bounds.append(second(e1) + c * second(a1 + e1))
    return np.maximum(bounds[0], bounds[1]) + 2.0 ** -45 * along_w(along_h(x))


def fp32_position_bound(x: np.ndarray, scale: float) -> np.ndarray:
    """Per-pixel bound on |BasicSR imresize - matlab_resize| where BasicSR forms the sample positions and the weights in fp32
    (torch.linspace, fp32 cubic) and sums with fp32 matrix-vector products in an unspecified order.

    Per output: u = x/scale + 0.5 (1 - 1/scale) and d = u - index carry at most 6 fp32 roundings of magnitude <= |u| + 2 width, so
    |delta d| <= dd = 6 u (|u|max + 2 width).  The cubic is Lipschitz with constant 25/18 and its fp32 evaluation (12 operations on
    terms of magnitude <= 24) errs by <= 12 * 24 u; with the antialias factor s (1 when upscaling) each raw weight errs by
    ew = s (25/18 s dd + 288 u).  Normalising by sum ~ 1 (>= 1/2 here) moves a weight by <= 2 ew + 4 |w| p ew + 2 u |w|.  A pass
    therefore errs by <= (2 ew p + (4 p ew + 2 u + gamma_2p) sum |w|) max|v|, the second pass carries the first's error through
    sum |w|, and the result adds matlab_bound."""
    x = np.asarray(x, dtype=np.float64)
    H, W = x.shape[-2], x.shape[-1]
    aa = scale < 1.0
    width = 4.0 / scale if aa else 4.0
    p = math.ceil(width) + 2
    s = scale if aa else 1.0
    umax = max(H, W) / scale + 1.0 + 2 * width
    dd = 6 * U32 * (umax + 2 * width)
    ew = s * (25.0 / 18.0 * s * dd + 288 * U32)
    wsum = max(np.abs(matlab_weights(n, scale)[0]).sum(axis=1).max() for n in (H, W))
    per_pass = 2 * ew * p + (4 * p * ew + 2 * U32 + _gamma(2 * p)) * wsum
    vmax = float(np.abs(x).max()) if x.size else 0.0
    e1 = per_pass * vmax
    e2 = wsum * e1 + per_pass * (wsum * vmax + e1)
    return matlab_bound(x, scale) + e2


# ---- inputs -------------------------------------------------------------------------------------------------------------------------
def image_u8(kind: str, h: int, w: int, c: int, seed: int) -> np.ndarray:
    """Seeded uint8 [h, w, c] image: 'random' (uniform noise, every sum and clip path) or 'smooth' (low-frequency gradients)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    if kind == "random":
        return rng.integers(0, 256, (h, w, c), dtype=np.uint8)
    yy, xx = np.meshgrid(np.arange(h, dtype=np.float64), np.arange(w, dtype=np.float64), indexing="ij")
    out = np.empty((h, w, c), np.float64)
    for ch in range(c):
        fy, fx, ph = rng.uniform(0.01, 0.08), rng.uniform(0.01, 0.08), rng.uniform(0, 2 * np.pi)
        out[:, :, ch] = 127.5 + 120 * np.sin(2 * np.pi * (fy * yy + fx * xx) + ph)
    return np.clip(np.rint(out), 0, 255).astype(np.uint8)


def image_f32(kind: str, b: int, c: int, h: int, w: int, seed: int) -> np.ndarray:
    """Seeded fp32 [b, c, h, w] in [0, 1]: 'random' (texture) or 'smooth'."""
    rng = np.random.Generator(np.random.PCG64(seed))
    if kind == "random":
        return rng.random((b, c, h, w), dtype=np.float32)
    yy, xx = np.meshgrid(np.arange(h, dtype=np.float64), np.arange(w, dtype=np.float64), indexing="ij")
    out = np.empty((b, c, h, w), np.float32)
    for i in range(b):
        for ch in range(c):
            fy, fx, ph = rng.uniform(1 / 256, 1 / 32), rng.uniform(1 / 256, 1 / 32), rng.uniform(0, 2 * np.pi)
            out[i, ch] = 0.5 + 0.45 * np.sin(2 * np.pi * (fy * yy + fx * xx) + ph)
    return out


# Pillow size pairs ((W, H) -> (W, H), Pillow's order): x2 / x3 / x4 down and up, non-integer ratios, 1 x n, more than 2x up
PIL_CASES = [((96, 72), (48, 36)), ((96, 72), (32, 24)), ((96, 72), (24, 18)), ((24, 18), (48, 36)), ((24, 18), (72, 54)),
             ((24, 18), (96, 72)), ((64, 48), (16, 12)), ((37, 53), (100, 17)), ((90, 60), (30, 20)), ((30, 20), (120, 80)),
             ((1, 40), (1, 13)), ((40, 1), (13, 1)), ((51, 77), (17, 25)), ((17, 25), (51, 75)), ((64, 64), (64, 21)),
             ((5, 7), (200, 3)), ((33, 29), (33, 29))]
