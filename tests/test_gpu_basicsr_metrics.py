"""`hitsir_b200.psnr_ssim_basicsr` (CUDA kernels behind `hitsir_psnr_ssim_basicsr`) against the extended-precision BasicSR scores of
tests/basicsr_ref.py within the bound derived there, the rounding conversion of `to_uint8_hwc(rounding="nearest")`, and
`evaluate(protocol="basicsr")`."""
import ctypes

import numpy as np
import pytest
import torch

from tests import basicsr_ref as R

pytestmark = pytest.mark.gpu

KINDS = ["random", "smooth", "flat0", "flat255"]


def _mse_ssim(sr_u8, hr_u8, crop, y):
    """The C entry's raw (mse, ssim) of two uint8 (B,H,W,3) numpy batches."""
    from hitsir_b200 import _capi
    lib = _capi.load()
    s, h = torch.from_numpy(sr_u8).cuda(), torch.from_numpy(hr_u8).cuda()
    B, H, W, _ = sr_u8.shape
    scratch = torch.empty(int(lib.hitsir_basicsr_metrics_scratch_doubles(B, H, W, crop, int(y))), dtype=torch.float64, device="cuda")
    mse = torch.empty(B, dtype=torch.float64, device="cuda")
    ssim = torch.empty(B, dtype=torch.float64, device="cuda")
    _capi.check(lib.hitsir_psnr_ssim_basicsr(ctypes.c_void_p(s.data_ptr()), ctypes.c_void_p(h.data_ptr()), B, H, W, crop, int(y),
                                             ctypes.c_void_p(scratch.data_ptr()), ctypes.c_void_p(mse.data_ptr()),
                                             ctypes.c_void_p(ssim.data_ptr()), None))
    return mse.cpu().numpy(), ssim.cpu().numpy()


def _check(sr_u8, hr_u8, crop, y):
    import hitsir_b200
    mse, ssim = _mse_ssim(sr_u8, hr_u8, crop, y)
    want_mse, mse_b, want, bound = R.psnr_ssim_exact(sr_u8, hr_u8, crop, y)
    assert np.all(np.abs(ssim - want) <= bound), (crop, y, ssim - want, bound)
    assert np.all(np.abs(mse - want_mse) <= mse_b), (crop, y, mse - want_mse, mse_b)
    if not y:
        for i in range(len(mse)):       # integer squares summed exactly: numpy's mean bit for bit
            assert mse[i] == R.mse_basicsr(R.bgr(sr_u8[i]), R.bgr(hr_u8[i]), crop, False)
    psnr, ssim2 = hitsir_b200.psnr_ssim_basicsr(torch.from_numpy(sr_u8).cuda(), torch.from_numpy(hr_u8).cuda(), crop, y)
    assert psnr.dtype == torch.float64 and psnr.shape == (len(mse),) and np.array_equal(ssim2.cpu().numpy(), ssim)
    assert np.allclose(psnr.cpu().numpy(), 10 * np.log10(65025.0 / mse), rtol=1e-14, atol=0)


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("crop", [0, 1, 4, 8])
@pytest.mark.parametrize("y", [True, False])
def test_small_and_medium_shapes_within_bound(kind, crop, y):
    for B, H, W in [(1, 2 * crop + 11, 2 * crop + 11), (3, 2 * crop + 12, 2 * crop + 45), (2, 100, 77), (1, 256, 200)]:
        sr, hr = R.inputs(kind, B, H, W, seed=H * 7 + W + crop)
        _check(R.tensor2img(sr), hr, crop, y)


@pytest.mark.parametrize("shape,kind,y", [((1, 1356, 2040), "smooth", True), ((1, 1356, 2040), "random", False),
                                          ((2, 1024, 1024), "flat255", True)])
def test_large_shapes_within_bound(shape, kind, y):
    B, H, W = shape
    sr, hr = R.inputs(kind, B, H, W, seed=5)
    _check(R.tensor2img(sr), hr, 4, y)


@pytest.mark.parametrize("y", [True, False])
def test_identical_deterministic_batch_independent_and_graph_capturable(y):
    import hitsir_b200
    sr, hr = R.inputs("smooth", 3, 70, 90, 11)
    s, h = torch.from_numpy(R.tensor2img(sr)).cuda(), torch.from_numpy(hr).cuda()
    p, q = hitsir_b200.psnr_ssim_basicsr(h, h, 4, y)
    assert torch.all(p == float("inf")) and torch.all(q == 1.0)
    first = hitsir_b200.psnr_ssim_basicsr(s, h, 4, y)
    again = hitsir_b200.psnr_ssim_basicsr(s, h, 4, y)
    assert all(torch.equal(a, b) for a, b in zip(first, again))
    for i in range(3):
        one = hitsir_b200.psnr_ssim_basicsr(s[i:i + 1], h[i:i + 1], 4, y)
        assert one[0][0] == first[0][i] and one[1][0] == first[1][i]
    torch.cuda.synchronize()
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        hitsir_b200.psnr_ssim_basicsr(s, h, 4, y)          # warm-up on the capture stream
    st.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=st):
        out = hitsir_b200.psnr_ssim_basicsr(s, h, 4, y)
    g.replay()
    torch.cuda.synchronize()
    assert all(torch.equal(a, b) for a, b in zip(out, first))


def test_rounding_conversion_matches_torch_round():
    import hitsir_b200
    g = torch.Generator().manual_seed(3)
    x = torch.rand(2, 3, 33, 47, generator=g) * 1.4 - 0.2
    # exact .5 ties: for each k an fp32 x whose fp32 product with 255 is k + 0.5
    ties = []
    for k in range(255):
        cand, lo, hi = [np.float32((k + 0.5) / 255)], np.float32((k + 0.5) / 255), np.float32((k + 0.5) / 255)
        for _ in range(8):
            lo, hi = np.nextafter(lo, np.float32(0)), np.nextafter(hi, np.float32(1))
            cand += [lo, hi]
        ties.append(float(next(c for c in cand if c * np.float32(255) == np.float32(k + 0.5))))
    assert len(ties) == 255
    x.view(-1)[:255] = torch.tensor(ties)
    x.view(-1)[255:258] = torch.tensor([-0.0, float("-inf"), float("inf")])
    xd = x.cuda()
    got = hitsir_b200.to_uint8_hwc(xd, rounding="nearest")
    want = (xd.clamp(0, 1) * 255).round().to(torch.uint8).permute(0, 2, 3, 1)
    assert torch.equal(got, want)
    assert np.array_equal(got.cpu().numpy(), R.tensor2img(x.numpy()))
    # the default stays the truncating conversion
    assert torch.equal(hitsir_b200.to_uint8_hwc(xd), (xd.clamp(0, 1) * 255).to(torch.uint8).permute(0, 2, 3, 1))
    with pytest.raises(ValueError):
        hitsir_b200.to_uint8_hwc(xd, rounding="floor")


def test_errors():
    import hitsir_b200
    from hitsir_b200 import _capi
    u = lambda *s: torch.zeros(*s, dtype=torch.uint8, device="cuda")     # noqa: E731
    with pytest.raises(ValueError):
        hitsir_b200.psnr_ssim_basicsr(u(1, 20, 20, 3), u(1, 20, 20, 3), 5)          # 20 - 10 < 11
    hitsir_b200.psnr_ssim_basicsr(u(1, 21, 21, 3), u(1, 21, 21, 3), 5)
    with pytest.raises(ValueError):
        hitsir_b200.psnr_ssim_basicsr(u(1, 30, 30, 3), u(1, 30, 31, 3), 0)
    with pytest.raises(ValueError):
        hitsir_b200.psnr_ssim_basicsr(u(1, 30, 30, 3), u(1, 30, 30, 3).float(), 0)
    with pytest.raises(ValueError):
        hitsir_b200.psnr_ssim_basicsr(u(1, 30, 30, 1), u(1, 30, 30, 1), 0)
    with pytest.raises(ValueError):
        hitsir_b200.psnr_ssim_basicsr(u(1, 30, 30, 3), u(1, 30, 30, 3), -1)
    with pytest.raises(RuntimeError):
        hitsir_b200.psnr_ssim_basicsr(u(1, 30, 30, 3), u(1, 30, 30, 3).cpu(), 0)
    lib = _capi.load()
    t = u(1, 30, 30, 3)
    out = torch.empty(2, dtype=torch.float64, device="cuda")
    p = ctypes.c_void_p
    assert lib.hitsir_psnr_ssim_basicsr(p(t.data_ptr()), p(t.data_ptr()), 1, 30, 30, 0, 1, None, p(out.data_ptr()), p(out.data_ptr()),
                                        None) == _capi.ERR_INVALID
    assert "null" in _capi.last_error()
    for args in [(0, 30, 30, 0), (1, 30, 30, -1), (1, 30, 20, 5), (1, 20, 30, 5)]:
        assert lib.hitsir_basicsr_metrics_scratch_doubles(*args, 1) == 0
        assert lib.hitsir_psnr_ssim_basicsr(p(t.data_ptr()), p(t.data_ptr()), *args, 1, p(out.data_ptr()), p(out.data_ptr()),
                                            p(out.data_ptr()), None) == _capi.ERR_INVALID


@pytest.fixture(scope="module")
def model():
    import hitsir_b200
    torch.manual_seed(0)
    return hitsir_b200.HiT_SIR(True, True, True, **hitsir_b200.PRO_KWARGS).eval().cuda()


@pytest.mark.parametrize("lr_kernel", ["pil", "matlab"])
@pytest.mark.parametrize("self_ensemble", [False, True])
@pytest.mark.parametrize("bicubic_baseline", [False, True])
@pytest.mark.parametrize("given_lr", [False, True])
def test_evaluate_basicsr_is_the_composition_of_public_calls(model, lr_kernel, self_ensemble, bicubic_baseline, given_lr):
    import hitsir_b200 as hb
    _, hr = R.inputs("smooth", 2, 160, 144, 60)
    hr_u8 = torch.from_numpy(hr).cuda()
    hr_f = hb.to_float_nchw(hr_u8)
    lr_given = torch.from_numpy(R.inputs("random", 2, 40, 36, 61)[1]).cuda() if given_lr else None
    got = hb.evaluate(model, hr_u8, lr_kernel=lr_kernel, self_ensemble=self_ensemble, bicubic_baseline=bicubic_baseline,
                      protocol="basicsr", lr_u8=lr_given)
    if given_lr:
        lr_u8 = lr_given
        lr = hb.to_float_nchw(lr_u8)
    elif lr_kernel == "pil":
        lr_u8 = hb.resize_bicubic(hr_u8, size=(40, 36))
        lr = hb.to_float_nchw(lr_u8)
    else:
        lr = hb.resize_bicubic(hr_f, scale=0.25, kernel="matlab")
    if lr_kernel == "pil":
        up = hb.to_float_nchw(hb.resize_bicubic(lr_u8, size=(160, 144)))
    else:
        up = hb.resize_bicubic(lr, scale=4.0, kernel="matlab")
    with torch.no_grad():
        sr = model.forward_x8(lr) if self_ensemble else model(lr)
    score = lambda y: hb.psnr_ssim_basicsr(hb.to_uint8_hwc(y, rounding="nearest"), hr_u8, 4, test_y_channel=True)     # noqa: E731
    want = dict(zip(("psnr_y", "ssim_y"), score(sr)))
    if bicubic_baseline:
        want["bicubic_psnr_y"], want["bicubic_ssim_y"] = score(up)
    assert set(got) == set(want)
    for k in want:
        assert got[k].dtype == torch.float64 and got[k].shape == (2,)
        assert torch.equal(got[k], want[k]), k
    # an explicit crop_border is passed through
    with torch.no_grad():
        sr1 = model(lr)
    c2 = hb.evaluate(model, hr_u8, lr_kernel=lr_kernel, protocol="basicsr", crop_border=2, lr_u8=lr_given)
    assert torch.equal(c2["ssim_y"], hb.psnr_ssim_basicsr(hb.to_uint8_hwc(sr1, rounding="nearest"), hr_u8, 2)[1])
    if given_lr:
        # the skimage protocol takes lr_u8 too
        sk = hb.evaluate(model, hr_u8, lr_kernel=lr_kernel, lr_u8=lr_given)
        assert torch.equal(sk["psnr_y"], hb.psnr_y(sr1, hr_f)) and torch.equal(sk["ssim_y"], hb.ssim_y(sr1, hr_f))


def test_evaluate_basicsr_errors(model):
    import hitsir_b200 as hb
    hr_u8 = torch.from_numpy(R.inputs("smooth", 1, 160, 144, 1)[1]).cuda()
    with pytest.raises(ValueError):
        hb.evaluate(model, hr_u8, protocol="basicsr", gaussian_weights=True)
    with pytest.raises(ValueError):
        hb.evaluate(model, hr_u8, protocol="basicsr", use_sample_covariance=False)
    with pytest.raises(ValueError):
        hb.evaluate(model, hr_u8, protocol="matlab")
    with pytest.raises(ValueError):
        hb.evaluate(model, hr_u8, crop_border=4)                      # the skimage protocol does not crop
    with pytest.raises(ValueError):
        hb.evaluate(model, hr_u8, protocol="basicsr", crop_border=67)  # 144 - 134 < 11
    with pytest.raises(ValueError):
        hb.evaluate(model, hr_u8, protocol="basicsr", crop_border=-1)
    for bad in [torch.zeros(1, 40, 40, 3, dtype=torch.uint8, device="cuda"), torch.zeros(1, 40, 36, 3, device="cuda"),
                torch.zeros(2, 40, 36, 3, dtype=torch.uint8, device="cuda"), torch.zeros(1, 40, 36, 3, dtype=torch.uint8)]:
        with pytest.raises(ValueError):
            hb.evaluate(model, hr_u8, protocol="basicsr", lr_u8=bad)
    out = hb.evaluate(model, hr_u8, protocol="basicsr", crop_border=66)  # 144 - 132 = 12: the smallest crop window that fits
    assert torch.isfinite(out["ssim_y"]).all()
