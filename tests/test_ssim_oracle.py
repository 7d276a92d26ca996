"""CPU checks of the Y-channel SSIM oracle (tests/ssim_ref.py): known answers, an independent direct-loop evaluation, the derived
error bound (covers the float32 restatement of skimage, is small, and rejects plausible mistakes), and the reference's own call."""
import ast
import os

import numpy as np
import pytest

from tests import ssim_ref as R

WINDOWS = [(False, True), (False, False), (True, True), (True, False)]     # (gaussian_weights, use_sample_covariance)


@pytest.mark.parametrize("gaussian,sample_cov", WINDOWS)
def test_identical_images_give_exactly_one(gaussian, sample_cov):
    sr, hr = R.inputs("random", 2, 23, 31, 1)
    assert np.all(R.ssim_y(hr, hr, True, gaussian, sample_cov) == 1.0)
    v, b = R.ssim_y_exact(hr, hr, True, gaussian, sample_cov)
    assert np.all(np.abs(v - 1.0) <= b)


@pytest.mark.parametrize("gaussian,sample_cov", WINDOWS)
def test_constant_images_closed_form(gaussian, sample_cov):
    a, b = np.float32(0.3), np.float32(0.7)
    hr = np.full((1, 3, 17, 19), a, np.float32)
    sr = np.full((1, 3, 17, 19), b, np.float32)
    ya = float(R.y_channel(hr)[0, 0, 0])
    yb = float(R.y_channel(sr)[0, 0, 0])
    want = (2 * ya * yb + R.C1) / (ya * ya + yb * yb + R.C1)
    v, bound = R.ssim_y_exact(sr, hr, True, gaussian, sample_cov)
    assert abs(v[0] - want) < 1e-12
    assert abs(R.ssim_y(sr, hr, True, gaussian, sample_cov)[0] - want) <= bound[0]


@pytest.mark.parametrize("gaussian", [False, True])
def test_sample_covariance_changes_only_cn(gaussian):
    sr, hr = R.inputs("smooth", 1, 40, 44, 2)
    x, y = R.y_planes(sr, hr)
    x, y = x[0].astype(np.float64), y[0].astype(np.float64)
    ws = R.win_size(gaussian)
    cn = ws * ws / (ws * ws - 1)
    # the direct evaluation with cn forced to 1 under use_sample_covariance=True is use_sample_covariance=False
    s_true = R.ssim_direct(x, y, gaussian, True)
    s_false = R.ssim_direct(x, y, gaussian, False)
    assert s_true != s_false
    v_true = R.ssim_y_exact(sr, hr, True, gaussian, True)[0][0]
    v_false = R.ssim_y_exact(sr, hr, True, gaussian, False)[0][0]
    assert abs(v_true - s_true) < 1e-12 and abs(v_false - s_false) < 1e-12
    assert cn == (49 / 48 if not gaussian else 121 / 120)


@pytest.mark.parametrize("gaussian,sample_cov", WINDOWS)
def test_symmetric_without_clipping(gaussian, sample_cov):
    sr, hr = R.inputs("random", 2, 20, 27, 3)
    assert np.array_equal(R.ssim_y(sr, hr, False, gaussian, sample_cov), R.ssim_y(hr, sr, False, gaussian, sample_cov))


@pytest.mark.parametrize("gaussian,sample_cov", WINDOWS)
def test_direct_loop_agrees_with_oracle(gaussian, sample_cov):
    # explicit window sums, no scipy: pins the window's centring, its weights and the interior crop
    sr, hr = R.inputs("random", 1, 13 if not gaussian else 15, 17, 4)
    x, y = R.y_planes(sr, hr)
    direct = R.ssim_direct(x[0].astype(np.float64), y[0].astype(np.float64), gaussian, sample_cov)
    v, b = R.ssim_y_exact(sr, hr, True, gaussian, sample_cov)
    assert abs(v[0] - direct) < 1e-12
    assert abs(R.ssim_y(sr, hr, True, gaussian, sample_cov)[0] - direct) <= b[0]


# Bound size: a flat region near Y = 1 is where fp32 evaluation loses most.  There the window variances vanish, so B2 ~ C2 = 9e-4,
# and a second moment of ~0.83 carries up to 3 fp32 roundings: the worst case is ~8e-4 per pixel (skimage's actual error reaches
# ~2e-4 there).  'flat1' has a quarter of the image flat near 1; 'smooth' varies over 48-128 pixels, so the variance is mostly sr's noise.
MAX_BOUND = {"random": 1e-5, "smooth": 2e-4, "flat1": 4e-4}


@pytest.mark.parametrize("kind", ["random", "smooth", "flat1"])
@pytest.mark.parametrize("gaussian,sample_cov", WINDOWS)
@pytest.mark.parametrize("clip", [True, False])
def test_float32_oracle_within_bound(kind, gaussian, sample_cov, clip):
    sr, hr = R.inputs(kind, 2, 96, 128, 6)
    v, b = R.ssim_y_exact(sr, hr, clip, gaussian, sample_cov)
    got = R.ssim_y(sr, hr, clip, gaussian, sample_cov)
    assert np.all(np.abs(got - v) <= b), (got - v, b)
    assert np.all(b <= MAX_BOUND[kind]), b


def _mutants(sr, hr, gaussian):
    x, y = R.y_planes(sr, hr, True)
    xu, yu = R.y_planes(sr, hr, False)
    xb, yb = R.y_planes(sr, hr, True, channels=(2, 1, 0))
    return {
        "window shifted by one pixel": R.ssim_plane(x[0], y[0], gaussian, True, origin=1),
        "cn dropped": R.ssim_plane(x[0], y[0], gaussian, True, cov_norm_on=False),
        "crop omitted": R.ssim_plane(x[0], y[0], gaussian, True, crop=False),
        "sr not clipped": R.ssim_plane(xu[0], yu[0], gaussian, True),
        "Y from BGR": R.ssim_plane(xb[0], yb[0], gaussian, True),
    }


@pytest.mark.parametrize("gaussian", [False, True])
def test_mutants_fall_outside_bound(gaussian):
    sr, hr = R.inputs("flat1", 1, 64, 80, 5)
    v, b = R.ssim_y_exact(sr, hr, True, gaussian, True)
    for name, m in _mutants(sr, hr, gaussian).items():
        assert abs(m - v[0]) > b[0], (name, m, v[0], b[0])


def test_window_too_small_raises():
    sr, hr = R.inputs("random", 1, 10, 10, 7)
    R.ssim_y(sr[:, :, :7, :7], hr[:, :, :7, :7])
    with pytest.raises(ValueError):
        R.ssim_y(sr[:, :, :6, :], hr[:, :, :6, :])
    with pytest.raises(ValueError):
        R.ssim_y(sr, hr, gaussian_weights=True)


def test_reference_ssim_call_is_reproduced():
    """Every structural_similarity call of the reference's experiments/experiment.py passes what ssim_y reproduces: two positional
    images, data_range=1, gaussian_weights / use_sample_covariance absent or literal, nothing else."""
    from oracle.reference import reference_dir
    if reference_dir() is None:
        pytest.skip("HITSIR_REFERENCE_DIR does not name a checkout of the original project")
    path = os.path.join(reference_dir(), "experiments", "experiment.py")
    src = open(path).read()
    calls = []
    for node in ast.walk(ast.parse(src)):
        if isinstance(node, ast.Call):
            f = node.func
            name = f.attr if isinstance(f, ast.Attribute) else (f.id if isinstance(f, ast.Name) else "")
            if name.endswith("structural_similarity"):
                calls.append(node)
    assert calls, "no structural_similarity call found"
    for c in calls:
        # ast cannot tell whether the images are 2-D: the line is printed for a reader to check
        print(f"{path}:{c.lineno}: {ast.get_source_segment(src, c)}")
        assert len(c.args) == 2 and not any(isinstance(a, ast.Starred) for a in c.args)
        kw = {k.arg: k.value for k in c.keywords}
        assert None not in kw, "**kwargs in the call"
        assert set(kw) <= {"data_range", "gaussian_weights", "use_sample_covariance"}, set(kw)
        assert "data_range" in kw and isinstance(kw["data_range"], ast.Constant) and kw["data_range"].value == 1
        for k in ("gaussian_weights", "use_sample_covariance"):
            if k in kw:
                assert isinstance(kw[k], ast.Constant) and isinstance(kw[k].value, bool)
