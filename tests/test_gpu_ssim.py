"""`hitsir_b200.ssim_y` (CUDA kernel behind `hitsir_ssim_y`) against the float64 SSIM of tests/ssim_ref.py, within the bound derived
from the arithmetic there, and its exactness, determinism and error behaviour."""
import ctypes

import numpy as np
import pytest
import torch

from tests import ssim_ref as R

pytestmark = pytest.mark.gpu

SHAPES = [(3, 37, 53), (2, 256, 256), (1, 7, 7), (1, 11, 11), (1, 64, 4097), (1, 1356, 2040), (2, 1024, 1024)]
COMBOS = [(g, sc, clip) for g in (False, True) for sc in (True, False) for clip in (True, False)]


def _gpu(sr, hr, clip=True, gaussian=False, sample_cov=True):
    import hitsir_b200
    return hitsir_b200.ssim_y(torch.from_numpy(sr).cuda(), torch.from_numpy(hr).cuda(), clip, gaussian, sample_cov).cpu().numpy()


@pytest.mark.parametrize("kind", ["random", "smooth", "flat1"])
@pytest.mark.parametrize("shape", SHAPES)
def test_ssim_y_matches_exact_within_bound(shape, kind):
    B, H, W = shape
    sr, hr = R.inputs(kind, B, H, W, seed=B * 1000 + H + W)
    ran = 0
    for gaussian, sample_cov, clip in COMBOS:
        if min(H, W) < R.win_size(gaussian):
            continue
        got = _gpu(sr, hr, clip, gaussian, sample_cov)
        want, bound = R.ssim_y_exact(sr, hr, clip, gaussian, sample_cov)
        assert got.dtype == np.float64 and got.shape == (B,)
        assert np.all(np.abs(got - want) <= bound), (gaussian, sample_cov, clip, got - want, bound)
        f32 = R.ssim_y(sr, hr, clip, gaussian, sample_cov)
        assert np.all(np.abs(got - f32) <= 2 * bound), (gaussian, sample_cov, clip, got - f32, bound)
        ran += 1
    assert ran > 0


@pytest.mark.parametrize("gaussian,sample_cov", [(False, True), (False, False), (True, True), (True, False)])
def test_ssim_y_exact_one_constant_closed_form_and_determinism(gaussian, sample_cov):
    sr, hr = R.inputs("smooth", 3, 70, 90, 11)
    one = _gpu(hr, hr, True, gaussian, sample_cov)
    assert np.all(one == 1.0), one
    a = np.full((1, 3, 20, 24), 0.3, np.float32)
    b = np.full((1, 3, 20, 24), 0.7, np.float32)
    want, bound = R.ssim_y_exact(b, a, True, gaussian, sample_cov)
    ya, yb = float(R.y_channel(a)[0, 0, 0]), float(R.y_channel(b)[0, 0, 0])
    assert abs(want[0] - (2 * ya * yb + R.C1) / (ya * ya + yb * yb + R.C1)) < 1e-12
    assert abs(_gpu(b, a, True, gaussian, sample_cov)[0] - want[0]) <= bound[0]
    # two calls are bit-identical, and an image's value does not depend on the rest of the batch
    first = _gpu(sr, hr, True, gaussian, sample_cov)
    assert np.array_equal(first, _gpu(sr, hr, True, gaussian, sample_cov))
    for i in range(3):
        assert _gpu(sr[i:i + 1], hr[i:i + 1], True, gaussian, sample_cov)[0] == first[i]


def test_ssim_y_on_model_output():
    # the eval loop of experiment.py without leaving the device: model -> clip -> Y -> SSIM against a synthetic ground truth
    import hitsir_b200
    model = hitsir_b200.HiT_SIR(True, True, True, **hitsir_b200.PRO_KWARGS).eval().cuda()
    x = torch.rand(2, 3, 40, 36, device="cuda")
    with torch.no_grad():
        sr = model(x)
    hr = (sr.detach().clamp(0, 1) + 0.05 * torch.randn_like(sr)).clamp(0, 1)
    srn, hrn = sr.cpu().numpy(), hr.cpu().numpy()
    for gaussian in (False, True):
        got = hitsir_b200.ssim_y(sr, hr, gaussian_weights=gaussian).cpu().numpy()
        want, bound = R.ssim_y_exact(srn, hrn, True, gaussian, True)
        assert np.all(np.abs(got - want) <= bound), (got - want, bound)


def test_ssim_y_errors():
    import hitsir_b200
    from hitsir_b200 import _capi
    with pytest.raises(RuntimeError):
        hitsir_b200.ssim_y(torch.zeros(1, 3, 8, 8), torch.zeros(1, 3, 8, 8))
    z = lambda *s: torch.zeros(*s, device="cuda")     # noqa: E731
    with pytest.raises(ValueError):
        hitsir_b200.ssim_y(z(1, 3, 6, 40), z(1, 3, 6, 40))
    with pytest.raises(ValueError):
        hitsir_b200.ssim_y(z(1, 3, 40, 10), z(1, 3, 40, 10), gaussian_weights=True)
    with pytest.raises(ValueError):
        hitsir_b200.ssim_y(z(1, 3, 16, 16), z(1, 3, 16, 17))
    with pytest.raises(ValueError):
        hitsir_b200.ssim_y(z(1, 1, 16, 16), z(1, 1, 16, 16))
    lib = _capi.load()
    t = z(1, 3, 16, 16)
    out = torch.empty(1, dtype=torch.float64, device="cuda")
    status = lib.hitsir_ssim_y(ctypes.c_void_p(t.data_ptr()), ctypes.c_void_p(t.data_ptr()), 1, 16, 16, 1, 0, 1, None,
                               ctypes.c_void_p(out.data_ptr()), None)
    assert status != 0 and "null" in _capi.last_error()
    assert lib.hitsir_ssim_y_scratch_doubles(1, 6, 16, 0) == 0
