"""CPU checks of the BasicSR PSNR / SSIM oracle (tests/basicsr_ref.py): the device's Y formula over every uint8 triple, the window
constants the kernel hard-codes, tensor2img's rounding, the cv2 restatement against the extended-precision reference within the
derived bound, mutants that the bound rejects, and the restatement against the vendored BasicSR itself when a checkout is at hand."""
import os
import re

import numpy as np
import pytest

from oracle.metrics import y_channel as y_skimage
from tests import basicsr_ref as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KINDS = ["random", "smooth", "flat0", "flat255"]


def test_device_order_y_equals_to_y_channel_for_all_triples():
    # y_basicsr's IEEE operation order (ycbcr.cuh) against BasicSR's to_y_channel, every (r, g, b), in four slabs of 2^22 pixels
    for slab in range(4):
        v = np.arange(slab << 22, (slab + 1) << 22, dtype=np.uint32)
        r, g, b = (v >> 16).astype(np.uint8), ((v >> 8) & 255).astype(np.uint8), (v & 255).astype(np.uint8)
        img_bgr = np.stack([b, g, r], axis=-1).reshape(2048, 2048, 3)
        want = R.to_y_channel(img_bgr)[..., 0].reshape(-1)
        got = R.y_device_order(r, g, b)
        assert want.dtype == got.dtype == np.float32
        assert np.array_equal(want.view(np.uint32), got.view(np.uint32)), slab


def test_window_constants_of_metrics_cu_are_cv2s():
    src = open(os.path.join(ROOT, "single-image-super-resolution-application_b200", "csrc", "metrics.cu")).read()
    body = re.search(r"kBsrGauss\[11\]\s*=\s*\{([^}]*)\}", src).group(1)
    taps = np.array([float.fromhex(t.strip()) for t in body.split(",")])
    assert np.array_equal(taps, R.KERNEL)
    assert np.abs(R.KERNEL - R.gaussian_formula()).max() < 1e-16
    # the kernel writes c1, c2 as (0.01 * 255) * (0.01 * 255); BasicSR as (0.01 * 255)**2
    assert R.C1 == (0.01 * 255) * (0.01 * 255) and R.C2 == (0.03 * 255) * (0.03 * 255)


def test_tensor2img_rounds_half_to_even_and_keeps_hr():
    # every uint8 HR value survives u8 / 255 -> tensor2img
    u = np.arange(256, dtype=np.uint8)
    x = (u.astype(np.float32) / np.float32(255)).reshape(1, 1, 1, 256)
    assert np.array_equal(R.tensor2img(x).reshape(-1), u)
    # for every k in 0..254 there are fp32 x with fp32(x * 255) == k + 0.5 exactly; tensor2img takes the even neighbour
    for k in range(255):
        x0 = np.float32((k + 0.5) / 255)
        cand, lo, hi = [x0], x0, x0
        for _ in range(8):
            lo, hi = np.nextafter(lo, np.float32(0)), np.nextafter(hi, np.float32(1))
            cand += [lo, hi]
        ties = [c for c in cand if np.float32(c) * np.float32(255) == np.float32(k + 0.5)]
        assert ties, k
        got = R.tensor2img(np.array(ties, np.float32).reshape(1, 1, 1, -1)).reshape(-1)
        assert np.all(got == (k if k % 2 == 0 else k + 1)), (k, got)
    # out of range clamps
    assert list(R.tensor2img(np.array([-0.5, 1.5, np.float32(-0.0)], np.float32).reshape(1, 1, 1, 3)).reshape(-1)) == [0, 255, 0]


@pytest.mark.parametrize("y", [True, False])
def test_identical_images(y):
    _, hr = R.inputs("smooth", 1, 40, 50, 1)
    p, s = R.psnr_ssim(hr, hr, 4, y)
    assert p[0] == float("inf") and s[0] == 1.0
    mse, _, v, b = R.psnr_ssim_exact(hr, hr, 4, y)
    assert mse[0] == 0 and abs(v[0] - 1.0) <= b[0]


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("y", [True, False])
@pytest.mark.parametrize("crop", [0, 4])
def test_cv2_restatement_within_bound(kind, y, crop):
    sr, hr = R.inputs(kind, 2, 64, 90, 2)
    su = R.tensor2img(sr)
    psnr, ssim = R.psnr_ssim(su, hr, crop, y)
    mse, mse_b, v, b = R.psnr_ssim_exact(su, hr, crop, y, dft=True)
    assert np.all(np.abs(ssim - v) <= b), (ssim - v, b)
    assert np.all(b < 1e-9), b
    for i in range(2):
        m = R.mse_basicsr(R.bgr(su[i]), R.bgr(hr[i]), crop, y)
        assert abs(m - mse[i]) <= mse_b[i]
        if not y:
            assert m == mse[i]                 # integer squares: numpy's mean is exact
        assert psnr[i] == 10. * np.log10(255. * 255. / m)


def test_mutants_fall_outside_bound():
    sr, hr = R.inputs("smooth", 1, 72, 96, 3)
    su = R.tensor2img(sr)
    c = 4
    mse, mse_b, v, b = R.psnr_ssim_exact(su, hr, c, True, dft=True)
    s, h = R.bgr(su[0]), R.bgr(hr[0])
    trunc = (np.clip(sr, 0, 1) * np.float32(255)).astype(np.uint8).transpose(0, 2, 3, 1)

    def ssim_planes(a, bb, **kw):
        return R._ssim(a.astype(np.float64), bb.astype(np.float64), **kw)

    def y_sk(img_rgb):            # the reference harness's Y (utils/utils.py:170-186) on BasicSR's 0-255 scale
        x = img_rgb.astype(np.float32).transpose(2, 0, 1)[None] / np.float32(255)
        return y_skimage(x)[0] * np.float32(255)

    ssim_mutants = {
        "crop 3": R.calculate_ssim(s, h, c - 1, True),
        "crop 5": R.calculate_ssim(s, h, c + 1, True),
        "R and B swapped": R.calculate_ssim(su[0], hr[0], c, True),
        "skimage's Y": ssim_planes(y_sk(su[0])[c:-c, c:-c], y_sk(hr[0])[c:-c, c:-c]),
        "truncating tensor2img": R.calculate_ssim(R.bgr(trunc[0]), h, c, True),
        "uniform 7x7 window": R.calculate_ssim(s, h, c, True, window=np.full((7, 7), 1 / 49)),
        "sample covariance": R.calculate_ssim(s, h, c, True, cn=121 / 120),
        "mean over 'same'": R.calculate_ssim(s, h, c, True, valid=False),
        "c1, c2 on [0, 1]": R.calculate_ssim(s, h, c, True, c1=0.01 ** 2, c2=0.03 ** 2),
    }
    for name, m in ssim_mutants.items():
        assert abs(m - v[0]) > b[0], (name, m, v[0], b[0])
    mse_mutants = {
        "crop 3": R.mse_basicsr(s, h, c - 1, True),
        "crop 5": R.mse_basicsr(s, h, c + 1, True),
        "R and B swapped": R.mse_basicsr(su[0], hr[0], c, True),
        "truncating tensor2img": R.mse_basicsr(R.bgr(trunc[0]), h, c, True),
        "RGB instead of Y": R.mse_basicsr(s, h, c, False),
    }
    for name, m in mse_mutants.items():
        assert abs(m - mse[0]) > mse_b[0], (name, m, mse[0], mse_b[0])


def test_vendored_basicsr_matches_restatement():
    """The restatement equals the vendored BasicSR's calculate_psnr / calculate_ssim bit for bit."""
    from oracle.reference import reference_dir
    root = reference_dir()
    if root is None:
        pytest.skip("HITSIR_REFERENCE_DIR does not name a checkout of the original project")
    if not os.path.exists(R.vendored_path(root)):
        pytest.skip(f"{R.vendored_path(root)} is not in the checkout")
    mod = R.load_vendored(root)
    for kind in ("random", "smooth", "flat255"):
        sr, hr = R.inputs(kind, 2, 48, 60, 9)
        su = R.tensor2img(sr)
        for i in range(2):
            s, h = R.bgr(su[i]), R.bgr(hr[i])
            for y in (True, False):
                for c in (0, 4):
                    assert mod.calculate_psnr(s, h, c, input_order="HWC", test_y_channel=y) == R.calculate_psnr(s, h, c, y)
                    assert mod.calculate_ssim(s, h, c, input_order="HWC", test_y_channel=y) == R.calculate_ssim(s, h, c, y)
