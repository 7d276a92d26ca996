"""CPU tests: pin the oracle to the reference's golden vectors, and the drop-in's parameter tree to the
reference's state_dict.  (Parity of the CUDA path itself is in test_gpu_parity.py, -m gpu.)"""
import os

import numpy as np
import pytest
import torch

import hitsir_b200
from oracle.weights import synthetic_image
from oracle.reference import reference_dir
from tests.helpers import GOLDEN_CASES, build_pair, load_golden


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_oracle_matches_reference_golden(name):
    g, meta = load_golden(name)
    model, oracle = build_pair(meta["flags"], meta["upsampler"], meta["upscale"], meta["mode"], meta["wseed"])
    # parameter tree of the drop-in == reference state_dict (names, order, shapes, count)
    mine = "\n".join(f"{k} {tuple(v.shape)}" for k, v in model.state_dict().items())
    assert mine == str(g["keys"])
    assert sum(p.numel() for p in model.parameters()) == int(g["n_params"])
    assert len(list(model.buffers())) == 0
    x = synthetic_image(*meta["shape"], seed=meta["xseed"])
    taps = {}
    with torch.no_grad():
        y = oracle.forward(x, taps)
    ref = torch.from_numpy(g["y"])
    assert y.shape == ref.shape
    # fp32 restatement vs fp32 reference: only summation-order noise
    assert (y - ref).abs().max().item() < 2e-5
    stride = int(g["tap_stride"])
    checked = 0
    for key in g.files:
        if not key.startswith("tap_") or key == "tap_stride":
            continue
        t = taps[key[4:]].reshape(-1)[::stride]
        r = torch.from_numpy(g[key])
        assert t.shape == r.shape, key
        scale = r.abs().max().item() + 1e-6
        assert (t - r).abs().max().item() / scale < 1e-4, key
        checked += 1
    assert checked >= 15


def test_oracle_matches_reference_scc_parts():
    """SCC.forward piece by piece (SURVEY.md 8c-ii): pooled relative-position bias (6, L, Lb) of hit_sir_pro.py:477-503, S-SC (:458-513)
    and C-SC (:515-540) for all six window sizes, against values recorded from the unmodified reference (make_golden_r2.py scc)."""
    g, meta = load_golden("scc_parts_56x72")
    model, oracle = build_pair(meta["flags"], meta["upsampler"], meta["upscale"], meta["mode"], meta["wseed"])
    x = synthetic_image(*meta["shape"], seed=meta["xseed"])
    taps = {}
    with torch.no_grad():
        oracle.forward(x, taps)
    for j in range(6):
        scc = taps[f"block0.{j}.scc"]                       # (B,H,W,180) = [S-SC 90 | C-SC 90] (:596)
        for kind, part in (("ssc", scc[..., :90]), ("csc", scc[..., 90:])):
            ref = torch.from_numpy(g[f"{kind}{j}"])
            got = part.reshape(-1)[::meta["s_stride"]]
            assert got.shape == ref.shape
            assert (got - ref).abs().max().item() <= 2e-5 * (ref.abs().max().item() + 1e-6), (kind, j)
        bias = oracle.pooled_bias(0, j)
        assert list(bias.shape) == list(g[f"bias{j}_shape"])
        ref = torch.from_numpy(g[f"bias{j}"])
        assert (bias.reshape(-1)[::meta["b_stride"]] - ref).abs().max().item() < 2e-6, j


def test_oracle_matches_reference_single_channel():
    """in_chans = 1: no RGB mean (hit_sir_pro.py:1130-1131), one-channel conv_first / upsample head."""
    g, meta = load_golden("gray_x4_direct_40x44")
    model, oracle = build_pair(meta["flags"], meta["upsampler"], meta["upscale"], meta["mode"], meta["wseed"], in_chans=1)
    assert "\n".join(f"{k} {tuple(v.shape)}" for k, v in model.state_dict().items()) == str(g["keys"])
    x = synthetic_image(*meta["shape"], seed=meta["xseed"], chans=1)
    with torch.no_grad():
        y = oracle(x)
    ref = torch.from_numpy(g["y"])
    assert y.shape == ref.shape == (2, 1, 160, 176)
    assert (y - ref).abs().max().item() < 2e-5 * max(1.0, ref.abs().max().item())


VARIANT_CASES = ["var_3conv_x2_direct_40x44", "var_ape_x2_direct_40x40", "var_noupsampler_40x44"]


def build_variant(meta):
    return build_pair(meta["flags"], meta["upsampler"], meta["upscale"], meta["mode"], meta["wseed"], **meta["extra"])


@pytest.mark.parametrize("name", VARIANT_CASES)
def test_oracle_matches_reference_constructor_variants(name):
    """SURVEY.md 8f-4: resi_connection='3conv' (:913-918, :1224-1231), ape=True (:1187-1189, :1293-1294), upsampler=None (:1260-1262,
    :1335-1344): same state_dict keys as the reference, oracle == reference output."""
    g, meta = load_golden(name)
    model, oracle = build_variant(meta)
    assert "\n".join(f"{k} {tuple(v.shape)}" for k, v in model.state_dict().items()) == str(g["keys"])
    x = synthetic_image(*meta["shape"], seed=meta["xseed"])
    with torch.no_grad():
        y = oracle(x)
    ref = torch.from_numpy(g["y"])
    assert y.shape == ref.shape
    assert (y - ref).abs().max().item() < 2e-5 * max(1.0, ref.abs().max().item())


def test_save_pretrained_from_pretrained_round_trip(tmp_path):
    """PyTorchModelHubMixin (hit_sir_pro.py:9, 1065): save_pretrained / from_pretrained on a local directory restores the weights
    bit for bit (the constructor arguments are given again by the caller, exactly as with the reference class, whose signature has no
    serialisable config either)."""
    kw = dict(hitsir_b200.PRO_KWARGS)
    kw.update(depths=[2, 2], num_heads=[6, 6], upsampler="pixelshuffledirect", upscale=2)
    src = hitsir_b200.HiT_SIR(True, True, True, **kw)
    with torch.no_grad():
        for p in src.parameters():
            p.add_(torch.randn_like(p) * 0.01)
    src.save_pretrained(str(tmp_path / "ckpt"))
    dst = hitsir_b200.HiT_SIR.from_pretrained(str(tmp_path / "ckpt"), is_mult_size_conv_feat_extract=True, is_channel_spatial_attn=True,
                                              is_fusion=True, **kw)
    assert list(dst.state_dict()) == list(src.state_dict())
    for k, v in src.state_dict().items():
        assert torch.equal(v, dst.state_dict()[k]), k


BIG_CASES = ["big_cfg3_tile576_x2ps_init", "big_cfg3_tile576_x2ps_stress", "big_cfg4_512_x4_init", "big_cfg4_512_x4_stress"]


def check_big(y, g, tol_abs, min_psnr=None):
    """Compare a full-size output with the strided sample / crops / moments kept in a big_* fixture.  Returns (max-abs, psnr) over the
    compared values, normalised like tests.helpers.assert_close."""
    from tests.helpers import psnr
    scale = max(1.0, float(g["absmax"]))
    got = [y.reshape(-1)[::int(g["stride"])]]
    ref = [torch.from_numpy(g["sample"])]
    c = int(g["crop"])
    for i, (y0, x0) in enumerate(g["origins"]):
        got.append(y[0, :, y0:y0 + c, x0:x0 + c].reshape(-1))
        ref.append(torch.from_numpy(g[f"crop{i}"]).reshape(-1))
    got, ref = torch.cat(got), torch.cat(ref)
    assert got.shape == ref.shape and torch.isfinite(got).all()
    err = (got - ref).abs().max().item() / scale
    p = psnr(got / scale, ref / scale)
    assert err < tol_abs, (err, scale)
    if min_psnr is not None:
        assert p > min_psnr, p
    assert abs(y.double().mean().item() - float(g["mean"])) < max(tol_abs, 1e-3) * scale
    return err, p


@pytest.mark.skipif(os.environ.get("HITSIR_SLOW_TESTS") != "1", reason="minutes of CPU per case: HITSIR_SLOW_TESTS=1 to run")
@pytest.mark.parametrize("name", BIG_CASES)
def test_oracle_matches_reference_at_baseline_sizes(name):
    g, meta = load_golden(name)
    model, oracle = build_pair(meta["flags"], meta["upsampler"], meta["upscale"], meta["mode"], meta["wseed"])
    x = synthetic_image(*meta["shape"], seed=meta["xseed"])
    with torch.no_grad():
        y = oracle(x)
    check_big(y, g, 5e-5)


def test_known_answer_param_count():
    # logs/.../模型参数量.txt:1 of the reference: the one known-answer value that pins the architecture
    m = hitsir_b200.HiT_SIR(True, True, True, **hitsir_b200.PRO_KWARGS)
    assert sum(p.numel() for p in m.parameters() if p.requires_grad) == 10220014
    assert len(m.state_dict()) == 1650


@pytest.mark.skipif(reference_dir() is None, reason="HITSIR_REFERENCE_DIR does not name a checkout of the original project")
def test_oracle_matches_live_reference():
    import contextlib, io, sys, warnings
    warnings.filterwarnings("ignore")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    ref_root = reference_dir()
    sys.path.insert(0, os.path.join(root, "oracle", "ref_shim"))
    sys.path.insert(0, ref_root)
    try:
        with contextlib.redirect_stdout(io.StringIO()):
            from models.hit_sir_pro import HiT_SIR as RefHiT
            ref = RefHiT(True, True, True, **hitsir_b200.PRO_KWARGS).eval()
        model, oracle = build_pair((1, 1, 1), "nearest+conv", 4, "stress", 11)
        ref.load_state_dict(model.state_dict(), strict=True)
        x = synthetic_image(1, 37, 45, seed=5)          # needs reflect padding for every window size
        with torch.no_grad():
            assert (ref(x) - oracle(x)).abs().max().item() < 2e-5
    finally:
        sys.path.remove(ref_root)
        sys.modules.pop("models.hit_sir_pro", None)
        sys.modules.pop("models", None)


def test_oracle_edge_cases():
    model, oracle = build_pair((0, 0, 0), "pixelshuffledirect", 2, "init", 3)
    with pytest.raises(RuntimeError):               # 32x32 cannot be reflect-padded to window 64 (hit_sir_pro.py:672)
        oracle(torch.rand(1, 3, 32, 32))
    y = oracle(torch.rand(1, 3, 33, 33))
    assert y.shape == (1, 3, 66, 66)
    with pytest.raises(AssertionError):
        from oracle.hitsir_oracle import HiTSIROracle, OracleConfig
        HiTSIROracle(model.state_dict(), OracleConfig(False, False, False, upscale=2, upsampler="nearest+conv"))
