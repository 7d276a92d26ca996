"""Every covered CUDA stage in isolation against an fp64 evaluation of its own exact inputs (-m gpu).

Each test feeds one stage the values its kernel consumes -- an injection (`hitsir_set_inject`) or a tap (`hitsir_set_tap`) of the same
deterministic forward -- reads the stage's output tap and asserts, element by element, the a-priori bound of tests/stage_ref.py:
K * 2^-22 * M_acc + sum of 2^-8 * M_site over the stage's bf16 rounding sites + one ulp of the output type.  The rounding sites and
the derivation of each bound are in the docstrings of the stage functions in tests/stage_ref.py; tests/test_stage_ref.py shows on the
CPU that the simulated kernel passes and plausible mutants fail the same assertion.  Each check prints its worst |got - ref| / bound.

Trunk: B = 2, 98 x 146, stress weights, flags (1, 1, 1): 28 616 tokens = 224 GEMM tiles of 128 (the last holds 72 rows), 2 x 13 x 10
conv tiles of 16 x 8 with partial tiles on both axes, so every persistent CTA takes several tiles.  HR: LR 1 x 37 x 53 (x4: 266 HR tiles
of 16 x 8)."""
import pytest
import torch

from oracle.weights import synthetic_image
from tests import stage_ref as sr
from tests.helpers import build_pair

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TB, TH, TW = 2, 98, 146
C = 180


def tap(model, x, name, shape):
    """One forward that stops after producing `name`; returns the tap on the host as float32 of `shape`."""
    n = 1
    for s in shape:
        n *= s
    dst = torch.full((n,), float("nan"), device=DEV)
    model.set_tap(DEV, name, dst, stop=True)
    with torch.no_grad():
        model(x)
    torch.cuda.synchronize()
    model.set_tap(DEV, None)
    out = dst.cpu().view(*shape)
    assert not torch.isnan(out).any(), name
    return out


def trunk_model(edit=None):
    model, oracle = build_pair((1, 1, 1), "nearest+conv", 4, "stress", 21, edit=edit)
    return model.to(DEV), oracle.sd


@pytest.fixture(scope="module")
def trunk():
    model, sd = trunk_model()
    x = synthetic_image(TB, TH, TW, seed=4).to(DEV)
    return model, sd, x


def stream(model, x):
    """A realistic token stream to inject as a block input: the patch-embedded image of the same forward."""
    return tap(model, x, "embed", (TB, TH, TW, C))


# ---- entry LayerNorm and the final LayerNorm ---------------------------------------------------------------------------------
@pytest.mark.parametrize("shift", [0.0, 512.0])
def test_ln_rows_patch_embed(shift):
    """`ln_rows` on the shallow features (tap `shallow` -> tap `embed`), fp32 in and out.  shift = 512 adds 512 to
    conv_first.conv_last.bias, so every row has |mean| >> std."""
    def edit(sd):
        sd["conv_first.conv_last.bias"] += shift
    model, sd = trunk_model(edit)
    x = synthetic_image(TB, TH, TW, seed=4).to(DEV)
    s = tap(model, x, "shallow", (TB, TH, TW, C))
    got = tap(model, x, "embed", (TB, TH, TW, C))
    ref, bound = sr.ln_rows(s, sd["patch_embed.norm.weight"], sd["patch_embed.norm.bias"], sr.REF, False)
    sr.check_bound(f"ln_rows embed (+{shift:g})", got, ref, bound)


def test_final_norm_and_conv_after_body(trunk):
    """final `ln_rows` (tap `layer5` -> bf16 tap `norm`) and `conv_after_body` (K = 1620, fp32 out) from the bf16 `norm` map."""
    model, sd, x = trunk
    l5 = tap(model, x, "layer5", (TB, TH, TW, C))
    norm = tap(model, x, "norm", (TB, TH, TW, C))
    ref, bound = sr.ln_rows(l5, sd["norm.weight"], sd["norm.bias"], sr.REF, True)
    sr.check_bound("final norm", norm, ref, bound)
    got = tap(model, x, "conv_after_body", (TB, TH, TW, C))
    ref, bound = sr.conv3(norm, sd["conv_after_body.weight"], sd["conv_after_body.bias"], sr.REF)
    sr.check_bound("conv_after_body", got, ref, bound)


# ---- block stages ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("j", range(6))
def test_proj_norm1_residual(trunk, j):
    """proj + norm1 + residual: tap `block0.j.scc` (bf16) + the injected stream -> tap `block0.j.attn`."""
    model, sd, x = trunk
    src = stream(model, x)
    model.set_inject(DEV, f"block0.{j}.in", src.reshape(-1, C).to(DEV))
    try:
        scc = tap(model, x, f"block0.{j}.scc", (TB, TH, TW, C))
        got = tap(model, x, f"block0.{j}.attn", (TB, TH, TW, C))
    finally:
        model.set_inject(DEV, None)
    ref, bound = sr.proj_norm1(scc, src, sr.block_params(sd, 0, j), sr.REF)
    sr.check_bound(f"proj_norm1 block0.{j}", got, ref, bound)


def test_proj_norm1_large_mean():
    """The LayerNorm epilogue with proj.bias += 256: |mean| >> std in every row (Chan's merge of per-slice (mean, M2))."""
    def edit(sd):
        sd["layers.0.residual_group.blocks.0.correlation.proj.bias"] += 256.0
    model, sd = trunk_model(edit)
    x = synthetic_image(TB, TH, TW, seed=4).to(DEV)
    src = stream(model, x)
    model.set_inject(DEV, "block0.0.in", src.reshape(-1, C).to(DEV))
    try:
        scc = tap(model, x, "block0.0.scc", (TB, TH, TW, C))
        got = tap(model, x, "block0.0.attn", (TB, TH, TW, C))
    finally:
        model.set_inject(DEV, None)
    ref, bound = sr.proj_norm1(scc, src, sr.block_params(sd, 0, 0), sr.REF)
    sr.check_bound("proj_norm1 block0.0, proj.bias + 256", got, ref, bound)


def planted_fc1_edit(j):
    """fc1 of block 0.j identity-like (hidden o reads stream channel o % 180, scale 0.5 .. 4, bias 0): pre-activations sweep
    the GELU fit densely, out to |x| >= 9 where s = x^2 is clamped at 81."""
    def edit(sd):
        p = f"layers.0.residual_group.blocks.{j}.mlp.fc1."
        w = torch.zeros_like(sd[p + "weight"])
        o = torch.arange(w.shape[0])
        w[o, o % w.shape[1]] = 0.5 + 3.5 * o.float() / (w.shape[0] - 1)
        sd[p + "weight"], sd[p + "bias"] = w, torch.zeros_like(sd[p + "bias"])
    return edit


@pytest.mark.parametrize("j,planted", [(j, False) for j in range(6)] + [(2, True)])
def test_fc1_gelu(j, planted, trunk):
    """fc1 + GELU (resident weights): bf16 of tap `block0.j.attn` -> tap `block0.j.fc1` (360 channels, bf16).  Element-wise bound
    and the binned mean of (got - ref) over the pre-activation (a systematic GELU error cannot hide under the bf16 rounding)."""
    if planted:
        model, sd = trunk_model(planted_fc1_edit(j))
        x = synthetic_image(TB, TH, TW, seed=4).to(DEV)
    else:
        model, sd, x = trunk
    attn = tap(model, x, f"block0.{j}.attn", (TB, TH, TW, C))
    got = tap(model, x, f"block0.{j}.fc1", (TB, TH, TW, 2 * C))
    ref, bound, pre = sr.fc1_gelu(attn, sr.block_params(sd, 0, j), sr.REF)
    name = f"fc1 block0.{j}" + (" planted" if planted else "")
    sr.check_bound(name, got, ref, bound)
    sr.check_binned_mean(name, got, ref, pre, covers=9.0 if planted else 0.0)


@pytest.mark.parametrize("j", range(6))
def test_ffn_tail(trunk, j):
    """`ffn_tail`: tap `block0.j.fc1` (bf16 h1) + tap `block0.j.attn` (fp32 stream) -> tap `block0.j`."""
    model, sd, x = trunk
    h1 = tap(model, x, f"block0.{j}.fc1", (TB, TH, TW, 2 * C))
    attn = tap(model, x, f"block0.{j}.attn", (TB, TH, TW, C))
    got = tap(model, x, f"block0.{j}", (TB, TH, TW, C))
    ref, bound = sr.ffn_tail(h1, attn, sr.block_params(sd, 0, j), sr.REF)
    sr.check_bound(f"ffn_tail block0.{j}", got, ref, bound)


def test_layer_conv(trunk):
    """The last block's bf16 shadow (written by `ffn_tail`'s statistics warp) + the layer conv (K = 1620, + the layer input):
    inject `block0.0.in`, tap `block0.5` -> tap `layer0`.  The conv reads bf16(block0.5) -- a wrong shadow fails here."""
    model, sd, x = trunk
    src = stream(model, x)
    model.set_inject(DEV, "block0.0.in", src.reshape(-1, C).to(DEV))
    try:
        b5 = tap(model, x, "block0.5", (TB, TH, TW, C))
        got = tap(model, x, "layer0", (TB, TH, TW, C))
    finally:
        model.set_inject(DEV, None)
    ref, bound = sr.conv3(b5, sd["layers.0.conv.weight"], sd["layers.0.conv.bias"], sr.REF, res=src)
    sr.check_bound("layer0 conv", got, ref, bound)


# ---- HR stage ----------------------------------------------------------------------------------------------------------------
LB, LH, LW = 1, 37, 53


@pytest.fixture(scope="module")
def hr():
    model, oracle = build_pair((1, 1, 1), "nearest+conv", 4, "stress", 23)
    model = model.to(DEV)
    x = synthetic_image(LB, LH, LW, seed=5).to(DEV)
    g = torch.Generator().manual_seed(7)
    fused = torch.randn(LB, LH, LW, C, generator=g)
    model.set_inject(DEV, "fused", fused.reshape(-1, C).to(DEV))
    taps = {"fused": fused}
    taps["conv_before_upsample"] = tap(model, x, "conv_before_upsample", (LB, LH, LW, 64))
    taps["up1"] = tap(model, x, "up1", (LB, 2 * LH, 2 * LW, 64))
    taps["up2"] = tap(model, x, "up2", (LB, 4 * LH, 4 * LW, 64))
    taps["hr"] = tap(model, x, "hr", (LB, 4 * LH, 4 * LW, 64))
    with torch.no_grad():
        taps["output"] = model(x).cpu().permute(0, 2, 3, 1).contiguous()
    model.set_inject(DEV, None)
    return oracle.sd, taps


def test_conv_before_upsample(hr):
    """conv3 180 -> 64 + LeakyReLU(0.01), bf16 out: inject `fused` -> tap `conv_before_upsample`."""
    sd, t = hr
    ref, bound = sr.conv3(t["fused"], sd["conv_before_upsample.0.weight"], sd["conv_before_upsample.0.bias"], sr.REF, slope=0.01,
                          bf16_out=True)
    sr.check_bound("conv_before_upsample", t["conv_before_upsample"], ref, bound)


@pytest.mark.parametrize("src,dst,k", [("conv_before_upsample", "up1", "conv_up1"), ("up1", "up2", "conv_up2")])
def test_conv3_c64_up(hr, src, dst, k):
    """`conv3_c64_up_kernel` (bf16 phase filters, interleaving TMA stores): previous tap -> tap `up1` / `up2`."""
    sd, t = hr
    ref, bound = sr.conv_up(t[src], sd[k + ".weight"], sd[k + ".bias"], sr.REF)
    sr.check_bound(dst, t[dst], ref, bound)


def test_conv_hr_and_conv_last_fold(hr):
    """`conv3_c64_kernel` conv_hr (tap `up2` -> tap `hr`) and `conv_last_fold_kernel` (tap `hr` -> model output + mean, NCHW)."""
    sd, t = hr
    ref, bound = sr.conv3(t["up2"], sd["conv_hr.weight"], sd["conv_hr.bias"], sr.REF, slope=0.2, bf16_out=True)
    sr.check_bound("conv_hr", t["hr"], ref, bound)
    ref, bound = sr.conv_last(t["hr"], sd["conv_last.weight"], sd["conv_last.bias"], sr.REF)
    sr.check_bound("conv_last_fold", t["output"], ref, bound)


@pytest.mark.parametrize("up,scale", [("pixelshuffle", 2), ("pixelshuffle", 3), ("pixelshuffle", 4), ("pixelshuffledirect", 2),
                                      ("pixelshuffledirect", 3), ("pixelshuffledirect", 4), (None, 4)])
def test_reconstruction_heads(up, scale):
    """The other heads, fed an injected `fused` map (LR 37 x 53): 'pixelshuffle' from tap `conv_before_upsample` through the
    EPI_SHUFFLE_BF16 Upsample convs and conv_last to the model output; 'pixelshuffledirect' (EPI_SHUFFLE_NCHW) and upsampler=None
    (`res_img` epilogue) from the injected map to the model output."""
    model, oracle = build_pair((1, 1, 1), up, scale, "stress", 31)
    model, sd = model.to(DEV), oracle.sd
    x = synthetic_image(LB, LH, LW, seed=6).to(DEV)
    fused = torch.randn(LB, LH, LW, C, generator=torch.Generator().manual_seed(8))
    model.set_inject(DEV, "fused", fused.reshape(-1, C).to(DEV))
    try:
        u0 = tap(model, x, "conv_before_upsample", (LB, LH, LW, 64)) if up == "pixelshuffle" else None
        with torch.no_grad():
            got = model(x).cpu().permute(0, 2, 3, 1).contiguous()
    finally:
        model.set_inject(DEV, None)
    if up == "pixelshuffle":
        ref, bound = sr.head_pixelshuffle(u0, sd, scale, sr.REF)
    elif up == "pixelshuffledirect":
        ref, bound = sr.head_direct(fused, sd, scale, sr.REF)
    else:
        ref, bound = sr.head_none(fused, x.cpu().permute(0, 2, 3, 1), sd, sr.REF)
    sr.check_bound(f"head {up} x{scale}", got, ref, bound)


def test_resi_3conv():
    """resi_connection='3conv': the layer conv (inject `block0.0.in`, tap `block0.5` -> tap `layer0`) and conv_after_body
    (tap `norm` -> tap `conv_after_body`), each conv3 -> LReLU -> bf16, conv1x1 -> LReLU -> bf16, conv3 (+ residual)."""
    model, oracle = build_pair((1, 1, 1), "nearest+conv", 4, "stress", 21, resi_connection="3conv")
    model, sd = model.to(DEV), oracle.sd
    x = synthetic_image(TB, TH, TW, seed=4).to(DEV)
    src = stream(model, x)
    model.set_inject(DEV, "block0.0.in", src.reshape(-1, C).to(DEV))
    try:
        b5 = tap(model, x, "block0.5", (TB, TH, TW, C))
        got = tap(model, x, "layer0", (TB, TH, TW, C))
    finally:
        model.set_inject(DEV, None)
    ref, bound = sr.resi_3conv(b5, sd, "layers.0.conv.", sr.REF, res=src)
    sr.check_bound("3conv layer0", got, ref, bound)
    norm = tap(model, x, "norm", (TB, TH, TW, C))
    got = tap(model, x, "conv_after_body", (TB, TH, TW, C))
    ref, bound = sr.resi_3conv(norm, sd, "conv_after_body.", sr.REF)
    sr.check_bound("3conv conv_after_body", got, ref, bound)


def test_umma_direct_backend_is_rejected_by_the_product_library(trunk):
    """The direct-store epilogue needs the unfused FFN tail, which only the -DHITSIR_AB_PATHS test build has: the product library
    refuses the backend instead of failing every forward afterwards."""
    model, _, x = trunk
    with pytest.raises(Exception, match="umma_direct"):
        model.set_gemm_backend(DEV, "umma_direct")
    model.set_gemm_backend(DEV, "umma")
    assert tap(model, x, "shallow", (TB, TH, TW, C)).abs().sum() > 0
