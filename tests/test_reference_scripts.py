"""The reference's own inference script, UNCHANGED, on the drop-in module (-m gpu).

north_star: "... the same forward(x) contract, so test.py and experiments/*_experiment.py run unchanged".  `test_experiment.py`
(of the original project) is the reference's single-image demo: `from models.hit_sir_pro import HiT_SIR` (:8),
`create_model()` (:25-32), `load_model_weights()` of a harness-format checkpoint {'start_epoch','model',...} (:35-50), PIL -> [0,1]
tensor -> `model(lr.unsqueeze(0)).clip(0, 1)` (:75) -> PIL -> `.show()`; it calls `main(...)` at import time (:96).  The test
executes that file byte for byte (runpy) from a scratch directory that holds the image and the checkpoint at the relative paths the
script hard-codes, with exactly the two-line integration of INTEGRATION.md section 1 applied (the `models.hit_sir_pro` import
resolves to hitsir_b200) and `PIL.Image.Image.show` stubbed to capture the result, and compares the shown image with the CPU oracle.

The script comes from a checkout of the original project named by HITSIR_REFERENCE_DIR; without one the test skips.
`experiments/hitsir_pro_experiment.py` cannot be imported in this image at all (lpips and skimage are not installed), with or
without the drop-in, so only its constructor call (:15-26) is replayed.
"""
import os
import runpy
import sys
import types

import numpy as np
import pytest
import torch

import hitsir_b200
from oracle.weights import fill_state_dict, synthetic_image
from oracle.hitsir_oracle import HiTSIROracle, OracleConfig
from oracle.reference import reference_dir

CKPT = "weights/hitsir_pro_loss(l1)_mulsizeconvextract(True)_casa(True)_fusion_embed_dim(180)_len(depths)(6)_augment/best_psnr_ssim_lpips_model.pth"
IMG = "data/test/RealSRSet+5images/0014.jpg"


@pytest.mark.gpu
@pytest.mark.skipif(reference_dir() is None, reason="HITSIR_REFERENCE_DIR does not name a checkout of the original project")
def test_reference_test_experiment_runs_unchanged(tmp_path, monkeypatch):
    from PIL import Image
    ref_root = reference_dir()
    # the files the script hard-codes, relative to its working directory
    proto = hitsir_b200.HiT_SIR(True, True, True, **hitsir_b200.PRO_KWARGS)
    sd = fill_state_dict(proto.state_dict(), 77, "init")
    os.makedirs(tmp_path / os.path.dirname(CKPT))
    torch.save({"start_epoch": 301, "model": sd, "optimizer": {"state": {}, "param_groups": []}}, tmp_path / CKPT)
    os.makedirs(tmp_path / os.path.dirname(IMG))
    lr = (synthetic_image(1, 44, 56, seed=33)[0].permute(1, 2, 0) * 255.0).to(torch.uint8).numpy()
    Image.fromarray(lr).save(tmp_path / IMG, quality=95)
    # INTEGRATION.md section 1: `models.hit_sir_pro` is the drop-in; everything else the script imports is the reference's own
    pkg = types.ModuleType("models")
    pkg.__path__ = []
    monkeypatch.setitem(sys.modules, "models", pkg)
    monkeypatch.setitem(sys.modules, "models.hit_sir_pro", sys.modules["hitsir_b200.hit_sir_pro"])
    for name in [m for m in sys.modules if m == "utils" or m.startswith("utils.")]:
        monkeypatch.delitem(sys.modules, name)
    monkeypatch.syspath_prepend(ref_root)
    shown = []
    monkeypatch.setattr(Image.Image, "show", lambda self, *a, **k: shown.append(self.copy()))
    monkeypatch.chdir(tmp_path)
    runpy.run_path(os.path.join(ref_root, "test_experiment.py"), run_name="test_experiment")
    assert len(shown) == 1
    sr = np.asarray(shown[0])
    assert sr.shape == (44 * 4, 56 * 4, 3) and sr.dtype == np.uint8
    # the same pipeline on the CPU oracle: PIL decode -> to_tensor -> forward -> clip -> to_pil_image (value * 255, truncated)
    with Image.open(tmp_path / IMG) as im:
        x = torch.from_numpy(np.asarray(im.convert("RGB")).copy()).permute(2, 0, 1).float().div(255.0).unsqueeze(0)
    with torch.no_grad():
        ref = HiTSIROracle(sd, OracleConfig())(x).clip(0, 1)
    ref_u8 = (ref[0] * 255.0).to(torch.uint8).permute(1, 2, 0).numpy()
    diff = np.abs(sr.astype(np.int32) - ref_u8.astype(np.int32))
    assert diff.max() <= 1, diff.max()                 # bf16-operand path vs fp32 oracle: at most one grey level
    assert (diff > 0).mean() < 0.05


def test_experiment_constructor_call_is_accepted():
    """experiments/hitsir_pro_experiment.py:15-26 and hitsir_pro_gan_experiment.py:21-32 construct the generator with exactly these
    keyword arguments (values from main.py:26-32); `.to(device)`, `.eval()`, `.train()`, `.parameters()`, `.named_parameters()` and
    strict `load_state_dict` are what experiments/experiment.py uses (:205, :223, :420, :557)."""
    m = hitsir_b200.HiT_SIR(is_mult_size_conv_feat_extract=True, is_channel_spatial_attn=True, is_fusion=True, embed_dim=180,
                            base_win_size=[8, 8], depths=[6] * 6, num_heads=[6] * 6, mlp_ratio=2, upsampler="nearest+conv",
                            hier_win_ratios=[0.5, 1, 2, 4, 6, 8, 10, 12]).to(torch.device("cpu"))
    assert m.eval() is m and m.train() is m
    assert sum(p.numel() for _, p in m.named_parameters() if p.requires_grad) == 10220014
    m.load_state_dict({k: v.clone() for k, v in m.state_dict().items()}, strict=True)
