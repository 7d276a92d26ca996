"""CPU checks of the bicubic restatements (tests/resize_ref.py): the Pillow one against Pillow itself bit for bit, MATLAB known
answers, the fp32 error bound, mutants, and -- with a checkout of the original project -- its own `imresize` and the LR its
`ImageTransforms` synthesises."""
import inspect
import sys

import numpy as np
import pytest

from tests import resize_ref as R

Image = pytest.importorskip("PIL.Image")


def _pillow(img: np.ndarray, out_w: int, out_h: int) -> np.ndarray:
    return np.asarray(Image.fromarray(img).resize((out_w, out_h), Image.BICUBIC))


@pytest.mark.parametrize("mode", ["L", "RGB"])
@pytest.mark.parametrize("kind", ["random", "smooth"])
@pytest.mark.parametrize("case", R.PIL_CASES, ids=[f"{a[0]}x{a[1]}-{b[0]}x{b[1]}" for a, b in R.PIL_CASES])
def test_pil_restatement_is_bit_exact(case, kind, mode):
    (w, h), (ow, oh) = case
    c = 3 if mode == "RGB" else 1
    img = R.image_u8(kind, h, w, c, seed=h * 1000 + w + ow)
    img = img[:, :, 0] if mode == "L" else img
    assert Image.fromarray(img).mode == mode
    want = _pillow(img, ow, oh)
    got = R.pil_resize(img, oh, ow)
    assert got.dtype == np.uint8 and got.shape == want.shape
    assert np.array_equal(got, want), np.argwhere(got != want)[:5]


def test_pil_mutants_break_bit_exactness():
    # each mutant changes some pixel of a non-integer resize; an exact 2x upscale has coefficients that 16 bits still hold exactly
    img = R.image_u8("random", 53, 37, 3, seed=7)
    for oh, ow in ((17, 100), (13, 12)):
        want = _pillow(img, ow, oh)
        assert np.array_equal(R.pil_resize(img, oh, ow), want)
        for name, kw in {"a = -0.75": dict(a=-0.75), "16 precision bits": dict(precision_bits=16),
                         "vertical pass first": dict(vertical_first=True)}.items():
            assert not np.array_equal(R.pil_resize(img, oh, ow, **kw), want), (name, oh, ow)


def test_pil_coefficients_sum_to_one_in_fixed_point():
    # normalised in double and rounded per weight: the fixed-point sum is 2^22 up to one unit per tap
    for n_in, n_out in ((96, 24), (24, 96), (53, 17), (7, 200), (40, 13)):
        for xmin, k in R.pil_coeffs(n_in, n_out):
            assert xmin >= 0 and xmin + len(k) <= n_in
            assert abs(sum(k) - (1 << 22)) <= len(k)


# ---- MATLAB -------------------------------------------------------------------------------------------------------------------------
SCALES = [0.25, 1 / 3, 0.5, 0.37, 1.0, 2.0, 3.0, 4.0]


@pytest.mark.parametrize("scale", SCALES)
def test_matlab_constant_stays_constant(scale):
    x = np.full((1, 3, 23, 31), 0.625, np.float32)
    y = R.matlab_resize(x, scale)
    assert y.shape == (1, 3, R.matlab_out_size(23, scale), R.matlab_out_size(31, scale))
    assert np.all(np.abs(y - 0.625) <= 1e-14)


def test_matlab_scale_one_is_identity_within_bound():
    x = R.image_f32("random", 1, 3, 19, 26, 1)
    y = R.matlab_resize(x, 1.0)
    assert np.all(np.abs(y - x) <= R.matlab_bound(x, 1.0))
    assert np.array_equal(y, x.astype(np.float64))


@pytest.mark.parametrize("scale", [0.25, 1 / 3, 0.5, 0.37])
def test_matlab_downscale_weights(scale):
    w, idx = R.matlab_weights(101, scale)
    assert np.all(np.abs(w.sum(axis=1) - 1.0) <= 1e-14)
    # the antialiased kernel is 4 / scale input pixels wide; the all-zero first and last of the ceil(width) + 2 columns are dropped
    assert w.shape[1] == int(np.ceil(4 / scale))
    assert np.all(np.diff(idx, axis=1) == 1)


def test_matlab_mirror_hand_case():
    # x4 downscale of 10 samples: output 1 sits at u = 4 - 1.5 = 2.5 (1-based), the 18 taps start at floor(u - 8) = -6 (1-based);
    # the first (distance 8.5 * 0.25 > 2) and last (-8.5) are zero, which leaves 1-based -5 .. 10, i.e. 0-based -6 .. 9.  The
    # half-sample mirror maps -1 -> 0, -7 -> 6, 10 -> 9
    w, idx = R.matlab_weights(10, 0.25)
    assert w.shape == (3, 16)
    assert idx[0, 0] == -6 and idx[0, -1] == 9
    assert list(R.mirror(np.array([-7, -2, -1, 0, 9, 10, 11, 19, 20]), 10)) == [6, 1, 0, 0, 9, 9, 8, 0, 0]
    m = R.matlab_matrix(10, 0.25)
    assert np.all(np.abs(m.sum(axis=1) - 1.0) <= 1e-14)


@pytest.mark.parametrize("scale", [0.25, 0.5, 2.0, 4.0])
@pytest.mark.parametrize("kind", ["random", "smooth"])
def test_matlab_fp32_evaluation_within_bound(scale, kind):
    # an fp32 evaluation with fp32 weights (the arithmetic of the CUDA kernel), in both pass orders
    x = R.image_f32(kind, 1, 3, 40, 52, 3)
    ref = R.matlab_resize(x, scale)
    bound = R.matlab_bound(x, scale)
    mh32 = R.matlab_matrix(40, scale).astype(np.float32)
    mw32 = R.matlab_matrix(52, scale).astype(np.float32)
    h_first = np.einsum("oh,bchw->bcow", mh32, x) @ mw32.T
    w_first = np.einsum("oh,bchw->bcow", mh32, x @ mw32.T)
    for got in (h_first, w_first):
        assert got.dtype == np.float32
        assert np.all(np.abs(got - ref) <= bound)
    assert bound.max() < 1e-5


def test_matlab_mutants_fall_outside_bound():
    x = R.image_f32("random", 1, 3, 48, 56, 9)
    for scale in (0.25, 0.5, 2.0):
        ref = R.matlab_resize(x, scale)
        bound = R.matlab_bound(x, scale)
        mutants = {"a = -0.75": R.matlab_resize(x, scale, a=-0.75), "clamp instead of mirror": R.matlab_resize(x, scale, boundary="clamp")}
        if scale < 1:
            mutants["no antialias"] = R.matlab_resize(x, scale, antialias=False)
        for name, m in mutants.items():
            assert m.shape == ref.shape, name
            assert np.any(np.abs(m - ref) > bound), (name, scale)


# ---- the original project's own code ------------------------------------------------------------------------------------------------
def _reference_utils():
    from oracle.reference import reference_dir
    root = reference_dir()
    if root is None:
        pytest.skip("HITSIR_REFERENCE_DIR does not name a checkout of the original project")
    if root not in sys.path:
        sys.path.insert(0, root)
    import utils.utils as U
    return U


@pytest.mark.parametrize("scale", [0.25, 0.5])
def test_reference_imresize_within_bound(scale):
    import torch
    U = _reference_utils()
    x = R.image_f32("smooth", 1, 3, 64, 80, 11)
    y = U.imresize(torch.from_numpy(x[0]), scale)
    y = (y.numpy() if hasattr(y, "numpy") else np.asarray(y)).astype(np.float64)
    ref = R.matlab_resize(x, scale)[0]
    assert y.shape == ref.shape
    assert np.all(np.abs(y - ref) <= R.fp32_position_bound(x, scale)[0])


def test_reference_image_transforms_lr_is_pillow_bicubic():
    """The LR the original project's `ImageTransforms` synthesises for a test-split HR image: equal bit for bit to the Pillow
    resize, the default `lr_kernel` of `evaluate`."""
    U = _reference_utils()
    sig = inspect.signature(U.ImageTransforms)
    print("ImageTransforms", sig)
    known = {"split": "test", "crop_size": 96, "scaling_factor": 4, "lr_img_type": "pil", "hr_img_type": "pil"}
    missing = [n for n, p in sig.parameters.items() if p.default is inspect.Parameter.empty and n not in known]
    assert not missing, f"ImageTransforms{sig}: no value known for {missing}"
    t = U.ImageTransforms(**{n: v for n, v in known.items() if n in sig.parameters})
    hr = Image.fromarray(R.image_u8("smooth", 96, 128, 3, 21))
    lr, hr_out = t(hr)[:2]
    hr_np = np.asarray(hr_out) if isinstance(hr_out, Image.Image) else None
    lr_np = np.asarray(lr) if isinstance(lr, Image.Image) else None
    assert lr_np is not None and hr_np is not None, (type(lr), type(hr_out))
    want = R.pil_resize(hr_np, hr_np.shape[0] // 4, hr_np.shape[1] // 4)
    assert np.array_equal(lr_np, want)
