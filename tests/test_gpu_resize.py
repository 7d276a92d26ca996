"""`hitsir_b200.resize_bicubic` (CUDA kernels behind `hitsir_resize_u8_pil` / `hitsir_resize_f32_matlab`) against Pillow bit for
bit and against the float64 MATLAB restatement of tests/resize_ref.py within its derived bound; determinism, graph capture, errors,
and `evaluate` against the explicit composition of the public calls."""
import ctypes

import numpy as np
import pytest
import torch

from tests import resize_ref as R

pytestmark = pytest.mark.gpu
Image = pytest.importorskip("PIL.Image")


def _pillow(img: np.ndarray, out_w: int, out_h: int) -> np.ndarray:
    return np.asarray(Image.fromarray(img).resize((out_w, out_h), Image.BICUBIC))


def _pil_gpu(batch: np.ndarray, oh: int, ow: int) -> np.ndarray:
    import hitsir_b200
    return hitsir_b200.resize_bicubic(torch.from_numpy(batch).cuda(), size=(oh, ow), kernel="pil").cpu().numpy()


@pytest.mark.parametrize("mode", ["L", "RGB"])
@pytest.mark.parametrize("case", R.PIL_CASES, ids=[f"{a[0]}x{a[1]}-{b[0]}x{b[1]}" for a, b in R.PIL_CASES])
def test_pil_kernel_equals_pillow(case, mode):
    (w, h), (ow, oh) = case
    c = 3 if mode == "RGB" else 1
    imgs = np.stack([R.image_u8(kind, h, w, c, seed=h * 1000 + w + ow + i) for i, kind in enumerate(["random", "smooth", "random"])])
    got = _pil_gpu(imgs, oh, ow)
    assert got.shape == (3, oh, ow, c) and got.dtype == np.uint8
    for i in range(3):
        want = _pillow(imgs[i, :, :, 0] if c == 1 else imgs[i], ow, oh)
        assert np.array_equal(got[i, :, :, 0] if c == 1 else got[i], want), (i, np.argwhere((got[i, :, :, 0] if c == 1 else got[i]) != want)[:5])
        # a batch equals per-image calls
        assert np.array_equal(_pil_gpu(imgs[i:i + 1], oh, ow)[0], got[i])


# the last two run after smaller calls and need more than 48 KB of shared memory for their tap tables (downscales by ~100 and ~40)
@pytest.mark.parametrize("shape,oh,ow", [((1, 1356, 2040, 3), 339, 510), ((2, 256, 256, 3), 1024, 1024), ((1, 1000, 700, 1), 71, 333),
                                         ((1, 1356, 2040, 3), 13, 20), ((1, 2000, 1500, 1), 50, 37)])
def test_pil_kernel_large(shape, oh, ow):
    imgs = np.stack([R.image_u8("smooth" if i % 2 else "random", shape[1], shape[2], shape[3], seed=40 + i) for i in range(shape[0])])
    got = _pil_gpu(imgs, oh, ow)
    for i in range(shape[0]):
        src = imgs[i, :, :, 0] if shape[3] == 1 else imgs[i]
        want = _pillow(src, ow, oh)
        assert np.array_equal(got[i, :, :, 0] if shape[3] == 1 else got[i], want)


@pytest.mark.parametrize("scale", [0.25, 1 / 3, 0.5, 0.37, 1.0, 2.0, 3.0, 4.0])
@pytest.mark.parametrize("kind", ["random", "smooth"])
def test_matlab_kernel_within_bound(scale, kind):
    import hitsir_b200
    x = R.image_f32(kind, 2, 3, 37, 53, seed=int(scale * 100))
    got = hitsir_b200.resize_bicubic(torch.from_numpy(x).cuda(), scale=scale, kernel="matlab").cpu().numpy()
    ref = R.matlab_resize(x, scale)
    assert got.dtype == np.float32 and got.shape == ref.shape
    assert np.all(np.abs(got - ref) <= R.matlab_bound(x, scale)), np.abs(got - ref).max()
    if scale == 1.0:
        assert np.array_equal(got, x)


@pytest.mark.parametrize("kind", ["random", "smooth"])
@pytest.mark.parametrize("shape,scale", [((1, 3, 1356, 2040), 0.25), ((1, 1, 339, 510), 4.0), ((3, 1, 64, 1), 0.5)])
def test_matlab_kernel_large_within_bound(shape, scale, kind):
    import hitsir_b200
    x = R.image_f32(kind, *shape, seed=5)
    got = hitsir_b200.resize_bicubic(torch.from_numpy(x).cuda(), scale=scale, kernel="matlab").cpu().numpy()
    ref = R.matlab_resize(x, scale)
    assert np.all(np.abs(got - ref) <= R.matlab_bound(x, scale)), np.abs(got - ref).max()


def test_determinism_and_graph_capture():
    import hitsir_b200
    u8 = torch.from_numpy(np.stack([R.image_u8("random", 301, 203, 3, s) for s in range(2)])).cuda()
    f32 = torch.from_numpy(R.image_f32("random", 2, 3, 301, 203, 3)).cuda()
    calls = [lambda: hitsir_b200.resize_bicubic(u8, size=(77, 90), kernel="pil"),
             lambda: hitsir_b200.resize_bicubic(u8, size=(903, 406), kernel="pil"),
             lambda: hitsir_b200.resize_bicubic(f32, scale=0.25, kernel="matlab"),
             lambda: hitsir_b200.resize_bicubic(f32, scale=3.0, kernel="matlab")]
    for fn in calls:
        a, b = fn(), fn()
        assert torch.equal(a, b)
        fn()                     # warm-up outside the capture (first-launch attributes)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            out = fn()
        out.zero_()
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(out, a)


def test_errors():
    import hitsir_b200
    from hitsir_b200 import _capi
    u8 = torch.zeros(1, 8, 8, 3, dtype=torch.uint8, device="cuda")
    f32 = torch.zeros(1, 3, 8, 8, device="cuda")
    with pytest.raises(RuntimeError):
        hitsir_b200.resize_bicubic(u8.cpu(), size=(4, 4))
    with pytest.raises(ValueError):
        hitsir_b200.resize_bicubic(u8, size=(4, 4), kernel="lanczos")
    with pytest.raises(ValueError):
        hitsir_b200.resize_bicubic(torch.zeros(1, 8, 8, 2, dtype=torch.uint8, device="cuda"), size=(4, 4))
    with pytest.raises(ValueError):
        hitsir_b200.resize_bicubic(u8, size=(0, 4))
    with pytest.raises(ValueError):
        hitsir_b200.resize_bicubic(u8, scale=0.5)
    with pytest.raises(ValueError):
        hitsir_b200.resize_bicubic(f32, scale=0.5)                     # fp32 needs kernel="matlab"
    with pytest.raises(ValueError):
        hitsir_b200.resize_bicubic(f32, scale=-1.0, kernel="matlab")
    with pytest.raises(ValueError):
        hitsir_b200.resize_bicubic(u8, scale=0.5, kernel="matlab")
    with pytest.raises(RuntimeError):
        hitsir_b200.to_float_nchw(f32)
    with pytest.raises(_capi.HitsirError) as e:          # tap tables larger than a CTA's shared memory (a downscale by 400)
        hitsir_b200.resize_bicubic(torch.zeros(1, 1, 40000, 1, dtype=torch.uint8, device="cuda"), size=(1, 100))
    assert e.value.status == _capi.ERR_INVALID
    lib = _capi.load()
    p = lambda t: ctypes.c_void_p(t.data_ptr())      # noqa: E731
    scratch = torch.empty(1 << 20, dtype=torch.uint8, device="cuda")
    out_u8 = torch.empty(1, 4, 4, 3, dtype=torch.uint8, device="cuda")
    out_f = torch.empty(1, 3, 4, 4, device="cuda")
    assert lib.hitsir_resize_u8_pil(p(u8), p(out_u8), 1, 8, 8, 3, 4, 4, p(scratch), None) == 0
    cases = [lib.hitsir_resize_u8_pil(None, p(out_u8), 1, 8, 8, 3, 4, 4, p(scratch), None),
             lib.hitsir_resize_u8_pil(p(u8), p(out_u8), 1, 8, 8, 3, 4, 4, None, None),
             lib.hitsir_resize_u8_pil(p(u8), p(out_u8), 0, 8, 8, 3, 4, 4, p(scratch), None),
             lib.hitsir_resize_u8_pil(p(u8), p(out_u8), 1, 0, 8, 3, 4, 4, p(scratch), None),
             lib.hitsir_resize_u8_pil(p(u8), p(out_u8), 1, 8, 8, 3, 0, 4, p(scratch), None),
             lib.hitsir_resize_u8_pil(p(u8), p(out_u8), 1, 8, 8, 2, 4, 4, p(scratch), None),
             lib.hitsir_resize_f32_matlab(p(f32), None, 1, 3, 8, 8, 0.5, p(scratch), None),
             lib.hitsir_resize_f32_matlab(p(f32), p(out_f), 1, 4, 8, 8, 0.5, p(scratch), None),
             lib.hitsir_resize_f32_matlab(p(f32), p(out_f), 0, 3, 8, 8, 0.5, p(scratch), None),
             lib.hitsir_resize_f32_matlab(p(f32), p(out_f), 1, 3, 8, 8, 0.0, p(scratch), None),
             lib.hitsir_u8hwc_to_f32nchw(p(u8), None, 1, 3, 8, 8, None)]
    assert all(s == _capi.ERR_INVALID for s in cases), cases
    assert lib.hitsir_resize_scratch_bytes(2, 8, 8, 4, 4) == 0 and lib.hitsir_resize_scratch_bytes(0, 8, 8, 0, 4) == 0
    torch.cuda.synchronize()


def test_to_float_nchw_is_to_tensor():
    import hitsir_b200
    u8 = torch.from_numpy(np.stack([R.image_u8("random", 31, 45, 3, s) for s in range(2)])).cuda()
    got = hitsir_b200.to_float_nchw(u8)
    # to_tensor's true division by 255 (torch's CUDA division by a scalar multiplies by the reciprocal instead)
    want = np.ascontiguousarray(u8.cpu().numpy().transpose(0, 3, 1, 2)).astype(np.float32) / np.float32(255)
    assert np.array_equal(got.cpu().numpy(), want)
    assert torch.equal(hitsir_b200.to_uint8_hwc(got), u8)


@pytest.fixture(scope="module")
def model():
    import hitsir_b200
    torch.manual_seed(0)
    return hitsir_b200.HiT_SIR(True, True, True, **hitsir_b200.PRO_KWARGS).eval().cuda()


@pytest.mark.parametrize("lr_kernel", ["pil", "matlab"])
@pytest.mark.parametrize("self_ensemble", [False, True])
@pytest.mark.parametrize("bicubic_baseline", [False, True])
def test_evaluate_is_the_composition_of_public_calls(model, lr_kernel, self_ensemble, bicubic_baseline):
    import hitsir_b200 as hb
    hr_u8 = torch.from_numpy(np.stack([R.image_u8("smooth", 160, 144, 3, 60), R.image_u8("random", 160, 144, 3, 61)])).cuda()
    got = hb.evaluate(model, hr_u8, lr_kernel=lr_kernel, self_ensemble=self_ensemble, bicubic_baseline=bicubic_baseline)
    hr = hb.to_float_nchw(hr_u8)
    if lr_kernel == "pil":
        lr_u8 = hb.resize_bicubic(hr_u8, size=(40, 36))
        lr = hb.to_float_nchw(lr_u8)
        up = hb.to_float_nchw(hb.resize_bicubic(lr_u8, size=(160, 144)))
    else:
        lr = hb.resize_bicubic(hr, scale=0.25, kernel="matlab")
        up = hb.resize_bicubic(lr, scale=4.0, kernel="matlab")
    with torch.no_grad():
        sr = model.forward_x8(lr) if self_ensemble else model(lr)
    want = {"psnr_y": hb.psnr_y(sr, hr), "ssim_y": hb.ssim_y(sr, hr)}
    if bicubic_baseline:
        want["bicubic_psnr_y"], want["bicubic_ssim_y"] = hb.psnr_y(up, hr), hb.ssim_y(up, hr)
    assert set(got) == set(want)
    for k in want:
        assert got[k].dtype == torch.float64 and got[k].shape == (2,)
        assert torch.equal(got[k], want[k]), k
    if bicubic_baseline:
        assert torch.all(got["bicubic_psnr_y"] > 10)


def test_evaluate_lr_is_pillow_lr_and_shape_errors(model):
    import hitsir_b200 as hb
    hr = np.stack([R.image_u8("smooth", 160, 144, 3, 70), R.image_u8("random", 160, 144, 3, 71)])
    lr = hb.resize_bicubic(torch.from_numpy(hr).cuda(), size=(40, 36)).cpu().numpy()
    for i in range(2):
        assert np.array_equal(lr[i], _pillow(hr[i], 36, 40))
    with pytest.raises(ValueError):
        hb.evaluate(model, torch.from_numpy(hr[:, :158]).cuda())
    with pytest.raises(ValueError):
        hb.evaluate(model, torch.from_numpy(hr).cuda(), lr_kernel="bilinear")
