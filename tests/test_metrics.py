"""Evaluation metric around the path (SURVEY.md 8f-2): the numpy oracle is pinned bit for bit to the reference's own
`convert_image` output (tests/golden/metrics_y_channel.npz); the CUDA kernel behind `hitsir_psnr_y` is checked against the oracle."""
import os

import numpy as np
import pytest
import torch

from oracle import metrics as om

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "metrics_y_channel.npz")


def test_oracle_y_channel_matches_reference_golden_bit_exactly():
    g = np.load(GOLDEN)
    assert np.array_equal(om.y_channel(g["hr"]), g["y_hr"])
    assert np.array_equal(om.y_channel(np.clip(g["sr"], 0, 1)), g["y_sr_clipped"])


def test_oracle_matches_live_reference_when_present():
    from oracle.reference import reference_dir
    if reference_dir() is None:
        pytest.skip("HITSIR_REFERENCE_DIR does not name a checkout of the original project")
    import sys
    sys.path.insert(0, reference_dir())
    from utils.utils import convert_image
    x = np.random.Generator(np.random.PCG64(7)).random((2, 3, 19, 23), dtype=np.float32)
    y = convert_image(torch.from_numpy(x), source="[0,1]", target="y-channel", is_lr=False, is_lr_amplify=False, scaling_factor=4).numpy()
    assert np.array_equal(om.y_channel(x), y)


def test_oracle_psnr_properties():
    g = np.load(GOLDEN)
    hr, sr = g["hr"], g["sr"]
    p = om.psnr_y(sr, hr)
    assert p.shape == (3,) and np.all(np.isfinite(p)) and np.all(p > 20) and np.all(p < 40)
    assert np.all(np.isinf(om.psnr_y(hr, hr)))                                   # identical images: skimage returns inf too
    assert np.all(om.psnr_y(sr, hr, clip=True) >= om.psnr_y(sr, hr, clip=False))  # hr lies in [0,1]: clipping sr can only help
    # known answer: a constant offset of 0.1 in every channel moves Y by 0.1 * (65.738 + 129.057 + 25.064) / 256
    a = np.full((1, 3, 8, 8), 0.5, np.float32)
    dy = 0.1 * (65.738 + 129.057 + 25.064) / 256
    assert abs(om.psnr_y(a + np.float32(0.1), a)[0] - 10 * np.log10(1 / dy ** 2)) < 1e-4


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(3, 37, 53), (2, 256, 256), (1, 1, 1), (1, 64, 4097)])
def test_cuda_psnr_y_matches_oracle(shape):
    import hitsir_b200
    B, H, W = shape
    rng = np.random.Generator(np.random.PCG64(B * 1000 + H + W))
    hr = rng.random((B, 3, H, W), dtype=np.float32)
    sr = (hr + rng.normal(0.0, 0.03, hr.shape).astype(np.float32)).astype(np.float32)
    for clip in (True, False):
        want = om.mse_y(sr, hr, clip)
        got = hitsir_b200.mse_y(torch.from_numpy(sr).cuda(), torch.from_numpy(hr).cuda(), clip).cpu().numpy()
        # same fp32 arithmetic per pixel; only the order of the float64 sum differs
        assert np.allclose(got, want, rtol=1e-12, atol=0.0), (got, want)
    p = hitsir_b200.psnr_y(torch.from_numpy(sr).cuda(), torch.from_numpy(hr).cuda()).cpu().numpy()
    assert np.allclose(p, om.psnr_y(sr, hr), rtol=0, atol=1e-9)
    # deterministic and exact on identical inputs
    p2 = hitsir_b200.psnr_y(torch.from_numpy(sr).cuda(), torch.from_numpy(hr).cuda()).cpu().numpy()
    assert np.array_equal(p, p2)
    assert np.all(np.isinf(hitsir_b200.psnr_y(torch.from_numpy(hr).cuda(), torch.from_numpy(hr).cuda()).cpu().numpy()))


@pytest.mark.gpu
def test_cuda_psnr_y_on_golden_and_model_output():
    import hitsir_b200
    g = np.load(GOLDEN)
    got = hitsir_b200.psnr_y(torch.from_numpy(g["sr"]).cuda(), torch.from_numpy(g["hr"]).cuda()).cpu().numpy()
    assert np.allclose(got, om.psnr_y(g["sr"], g["hr"]), rtol=0, atol=1e-9)
    # the eval loop of experiment.py:743-755 without leaving the device: model -> clip -> Y -> PSNR against a synthetic ground truth
    model = hitsir_b200.HiT_SIR(True, True, True, **hitsir_b200.PRO_KWARGS).eval().cuda()
    x = torch.rand(2, 3, 40, 36, device="cuda")
    with torch.no_grad():
        sr = model(x)
    hr = torch.rand_like(sr)
    got = hitsir_b200.psnr_y(sr, hr).cpu().numpy()
    assert np.allclose(got, om.psnr_y(sr.cpu().numpy(), hr.cpu().numpy()), rtol=0, atol=1e-9)


def test_metrics_reject_cpu_tensors():
    import hitsir_b200
    with pytest.raises(RuntimeError):
        hitsir_b200.psnr_y(torch.zeros(1, 3, 4, 4), torch.zeros(1, 3, 4, 4))
