"""The stage references and bounds of tests/stage_ref.py, checked without a device.  Per stage:

(a) pinning: the fp64 stage function, fed the oracle's own fp32 operands, reproduces the oracle's tap to fp32 noise;
(b) the simulated kernel (fp32, bf16 operands, bf16 rounding at the kernel's sites) passes the bound: it is not tighter than the
    documented arithmetic;
(c) plausible kernel bugs applied to the simulated kernel are rejected by the same assertion: the bound is tight enough to matter.

tests/test_gpu_stage_fp64.py and tests/test_gpu_stage_fp64_front.py (window self-correlation, casa gate, entry, fusion) make the same assertions on the
CUDA kernels."""
import pytest
import torch

from oracle.weights import synthetic_image
from tests import stage_ref as sr
from tests.helpers import build_pair

B, H, W = 2, 33, 37


@pytest.fixture(scope="module")
def net():
    _, oracle = build_pair((1, 1, 1), "nearest+conv", 4, "stress", 21)
    taps = {}
    with torch.no_grad():
        y = oracle.forward(synthetic_image(B, H, W, seed=4), taps)
    taps["output"] = y.permute(0, 2, 3, 1).contiguous()
    return oracle.sd, taps


def fp32_noise(name, got, want, rel=2e-5):
    """|got - want| <= rel * max|want|: fp32 arithmetic against fp64 with the same operands."""
    err = (got.double() - want.double()).abs().max().item()
    scale = want.double().abs().max().item()
    assert err <= rel * scale, (name, err, scale)


def rejected(name, got, ref, bound):
    with pytest.raises(AssertionError):
        sr.check_bound(name, got, ref, bound)


def block_input(taps, j):
    return taps["embed"] if j == 0 else taps[f"block0.{j - 1}"]


# ---- ln_rows ------------------------------------------------------------------------------------------------------------------
def test_ln_rows(net):
    sd, taps = net
    g, b = sd["patch_embed.norm.weight"], sd["patch_embed.norm.bias"]
    fp32_noise("embed", sr.ln_rows(taps["shallow"], g, b, sr.PIN, False)[0], taps["embed"])
    fp32_noise("norm", sr.ln_rows(taps["layer5"], sd["norm.weight"], sd["norm.bias"], sr.PIN, False)[0], taps["norm"])
    for x, bf16_out in ((taps["shallow"], False), (taps["layer5"], True)):
        ref, bound = sr.ln_rows(x, g, b, sr.REF, bf16_out)
        sr.check_bound("ln_rows sim", sr.ln_rows(x, g, b, sr.SIM, bf16_out)[0], ref, bound)


def large_mean_rows(x):
    """Rows with |mean| >> std (the shallow features with conv_first.conv_last.bias += 512: a one-pass variance cancels there), and
    rows of a spread close to sqrt(eps) around 0 (where eps matters)."""
    x = x.clone() + 512.0
    x[:, ::3, :, :] = (x[:, ::3, :, :] - 512.0) * 3e-3
    return x


@pytest.mark.parametrize("mut", ["ln_eps", "ln_onepass"])
def test_ln_rows_mutants(net, mut):
    sd, taps = net
    g, b = sd["patch_embed.norm.weight"], sd["patch_embed.norm.bias"]
    x = large_mean_rows(taps["shallow"])
    ref, bound = sr.ln_rows(x, g, b, sr.REF, False)
    sr.check_bound("ln_rows sim, large mean", sr.ln_rows(x, g, b, sr.SIM, False)[0], ref, bound)
    rejected(mut, sr.ln_rows(x, g, b, sr.SIM, False, {mut})[0], ref, bound)


# ---- proj + norm1 + residual ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("j", range(6))
def test_proj_norm1(net, j):
    sd, taps = net
    P = sr.block_params(sd, 0, j)
    scc, xin = taps[f"block0.{j}.scc"], block_input(taps, j)
    fp32_noise("attn", sr.proj_norm1(scc, xin, P, sr.PIN)[0], taps[f"block0.{j}.attn"])
    ref, bound = sr.proj_norm1(scc, xin, P, sr.REF)
    sr.check_bound("proj_norm1 sim", sr.proj_norm1(scc, xin, P, sr.SIM)[0], ref, bound)
    rejected("res_bf16", sr.proj_norm1(scc, xin, P, sr.SIM, {"res_bf16"})[0], ref, bound)


def test_proj_norm1_large_mean_and_eps_mutant(net):
    """proj.bias += 256 (the GPU test's large-mean case): |mean| >> std in every LayerNorm row, and the simulated kernel still passes.
    proj scaled by 1e-3: the rows' variance is close to eps, and eps = 1e-6 is rejected.  (A one-pass fp32 variance is not rejected
    here: at |mean| / std ~ 256 it loses less than the worst-case bound of the mean's reduction allows; `ln_rows` rejects it.)"""
    sd, taps = net
    scc, xin = taps["block0.0.scc"], taps["embed"]
    P = dict(sr.block_params(sd, 0, 0))
    P["proj.bias"] = P["proj.bias"] + 256.0
    ref, bound = sr.proj_norm1(scc, xin, P, sr.REF)
    sr.check_bound("proj_norm1 sim, large mean", sr.proj_norm1(scc, xin, P, sr.SIM)[0], ref, bound)
    P = dict(sr.block_params(sd, 0, 0))
    P["proj.weight"], P["proj.bias"] = P["proj.weight"] * 1e-3, P["proj.bias"] * 1e-3
    ref, bound = sr.proj_norm1(scc, xin, P, sr.REF)
    sr.check_bound("proj_norm1 sim, small spread", sr.proj_norm1(scc, xin, P, sr.SIM)[0], ref, bound)
    rejected("ln_eps", sr.proj_norm1(scc, xin, P, sr.SIM, {"ln_eps"})[0], ref, bound)


# ---- fc1 + GELU ---------------------------------------------------------------------------------------------------------------
def planted_fc1(P):
    """Identity-like fc1: hidden channel o reads stream channel o % 180 with a scale growing from 0.5 to 4, bias 0, so the
    pre-activations sweep the GELU fit densely out to |x| >= 9 (where s = x^2 is clamped at 81)."""
    P = dict(P)
    w = torch.zeros_like(P["fc1.weight"])
    o = torch.arange(w.shape[0])
    w[o, o % w.shape[1]] = 0.5 + 3.5 * o.float() / (w.shape[0] - 1)
    P["fc1.weight"], P["fc1.bias"] = w, torch.zeros_like(P["fc1.bias"])
    return P


@pytest.mark.parametrize("planted", [False, True])
def test_fc1_gelu(net, planted):
    sd, taps = net
    P = sr.block_params(sd, 0, 2)
    attn = taps["block0.2.attn"]
    if planted:
        P = planted_fc1(P)
    pin = sr.fc1_gelu(attn, P, sr.PIN)[0]
    fp32_noise("fc1", pin, torch.nn.functional.gelu(torch.nn.functional.linear(attn, P["fc1.weight"], P["fc1.bias"])))
    ref, bound, pre = sr.fc1_gelu(attn, P, sr.REF)
    sim = sr.fc1_gelu(attn, P, sr.SIM)[0]
    sr.check_bound("fc1 sim", sim, ref, bound)
    sr.check_binned_mean("fc1 sim", sim, ref, pre, covers=9.0 if planted else 0.0)
    # x * sigmoid(1.702 x) differs from erf-GELU by up to 2e-2.  torch's tanh form (4.7e-4 at most) is not rejected: gelu2 itself
    # may be 2^-12 |x| away from erf-GELU (tanh.approx.f32), which is as large.
    sig = sr.fc1_gelu(attn, P, sr.SIM, {"gelu_sigmoid"})[0]
    with pytest.raises(AssertionError):
        sr.check_bound("gelu_sigmoid", sig, ref, bound)
        sr.check_binned_mean("gelu_sigmoid", sig, ref, pre)


# ---- FFN tail -----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("j", [0, 5])
def test_ffn_tail(net, j):
    sd, taps = net
    P = sr.block_params(sd, 0, j)
    attn = taps[f"block0.{j}.attn"]
    h1 = sr.fc1_gelu(attn, P, sr.PIN)[0]
    fp32_noise("block", sr.ffn_tail(h1, attn, P, sr.PIN)[0], taps[f"block0.{j}"])
    h1 = sr.bf(h1).float()                     # the kernel reads the bf16 fc1 output
    ref, bound = sr.ffn_tail(h1, attn, P, sr.REF)
    sr.check_bound("ffn_tail sim", sr.ffn_tail(h1, attn, P, sr.SIM)[0], ref, bound)
    rejected("dw_transposed", sr.ffn_tail(h1, attn, P, sr.SIM, {"dw_transposed"})[0], ref, bound)


# ---- 3x3 convs of the trunk ---------------------------------------------------------------------------------------------------
def test_layer_conv_and_conv_after_body(net):
    sd, taps = net
    w, b = sd["layers.0.conv.weight"], sd["layers.0.conv.bias"]
    fp32_noise("layer0", sr.conv3(taps["block0.5"], w, b, sr.PIN, res=taps["embed"])[0], taps["layer0"])
    ref, bound = sr.conv3(taps["block0.5"], w, b, sr.REF, res=taps["embed"])
    sr.check_bound("layer conv sim", sr.conv3(taps["block0.5"], w, b, sr.SIM, res=taps["embed"])[0], ref, bound)
    rejected("taps transposed", sr.conv3(taps["block0.5"], w.transpose(-1, -2).contiguous(), b, sr.SIM, res=taps["embed"])[0], ref, bound)
    w, b = sd["conv_after_body.weight"], sd["conv_after_body.bias"]
    fp32_noise("conv_after_body", sr.conv3(taps["norm"], w, b, sr.PIN)[0], taps["conv_after_body"])
    ref, bound = sr.conv3(sr.bf(taps["norm"]), w, b, sr.REF)
    sr.check_bound("conv_after_body sim", sr.conv3(taps["norm"], w, b, sr.SIM)[0], ref, bound)
    wt = w.transpose(-1, -2).contiguous()
    rejected("taps transposed", sr.conv3(taps["norm"], wt, b, sr.SIM)[0], ref, bound)


# ---- HR stage -----------------------------------------------------------------------------------------------------------------
def test_conv_before_upsample(net):
    sd, taps = net
    w, b = sd["conv_before_upsample.0.weight"], sd["conv_before_upsample.0.bias"]
    fp32_noise("cbu", sr.conv3(taps["fused"], w, b, sr.PIN, slope=0.01)[0], taps["conv_before_upsample"])
    ref, bound = sr.conv3(taps["fused"], w, b, sr.REF, slope=0.01, bf16_out=True)
    sr.check_bound("cbu sim", sr.conv3(taps["fused"], w, b, sr.SIM, slope=0.01, bf16_out=True)[0], ref, bound)
    rejected("lrelu 0.2", sr.conv3(taps["fused"], w, b, sr.SIM, slope=0.01, bf16_out=True, mut={"lrelu_slope"})[0], ref, bound)


@pytest.mark.parametrize("src,dst,k", [("conv_before_upsample", "up1", "conv_up1"), ("up1", "up2", "conv_up2")])
def test_conv_up(net, src, dst, k):
    sd, taps = net
    w, b = sd[k + ".weight"], sd[k + ".bias"]
    fp32_noise(dst, sr.conv_up(taps[src], w, b, sr.PIN)[0], taps[dst])
    x = sr.bf(taps[src]).float()
    ref, bound = sr.conv_up(x, w, b, sr.REF)
    sr.check_bound(dst + " sim", sr.conv_up(x, w, b, sr.SIM)[0], ref, bound)
    rejected("phases swapped", sr.conv_up(x, w, b, sr.SIM, {"phase_swap"})[0], ref, bound)


def test_conv_hr_and_conv_last(net):
    sd, taps = net
    w, b = sd["conv_hr.weight"], sd["conv_hr.bias"]
    fp32_noise("hr", sr.conv3(taps["up2"], w, b, sr.PIN, slope=0.2)[0], taps["hr"])
    x = sr.bf(taps["up2"]).float()
    ref, bound = sr.conv3(x, w, b, sr.REF, slope=0.2, bf16_out=True)
    sr.check_bound("hr sim", sr.conv3(x, w, b, sr.SIM, slope=0.2, bf16_out=True)[0], ref, bound)
    w, b = sd["conv_last.weight"], sd["conv_last.bias"]
    fp32_noise("output", sr.conv_last(taps["hr"], w, b, sr.PIN)[0], taps["output"])
    x = sr.bf(taps["hr"]).float()
    ref, bound = sr.conv_last(x, w, b, sr.REF)
    sr.check_bound("conv_last sim", sr.conv_last(x, w, b, sr.SIM)[0], ref, bound)
    rejected("taps transposed", sr.conv_last(x, w.transpose(-1, -2).contiguous(), b, sr.SIM)[0], ref, bound)


def test_ulp_and_bf16_rounding():
    assert sr.ulp(torch.tensor([1.0, 1.5, -3.0]), True).tolist() == [2.0 ** -7, 2.0 ** -7, 2.0 ** -6]
    assert sr.ulp(torch.tensor([1.0]), False).item() == 2.0 ** -23
    x = torch.tensor([1.0 + 2.0 ** -8, 1.0 + 3 * 2.0 ** -8])       # ties to even
    assert sr.bf(x).tolist() == [1.0, 1.0 + 2.0 ** -6]


def test_failure_names_the_worst_element():
    ref = torch.zeros(2, 3, 4, 5, dtype=torch.float64)
    got = ref.clone()
    got[1, 2, 0, 3] = 1.0
    with pytest.raises(AssertionError, match="image 1, y 2, x 0, channel 3"):
        sr.check_bound("t", got, ref, torch.full_like(ref, 0.5))


# ---- reconstruction heads and the 3conv residual connection ----------------------------------------------------------------------
def noise_map(*shape, seed, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(*shape, generator=g) * scale


@pytest.mark.parametrize("scale", [2, 3, 4])
def test_head_pixelshuffle(scale):
    _, oracle = build_pair((1, 1, 1), "pixelshuffle", scale, "stress", 31)
    sd = oracle.sd
    u0 = sr.bf(noise_map(2, 9, 11, 64, seed=scale).clamp_min(0)).float()        # conv_before_upsample output: LeakyReLU, bf16
    y = u0.permute(0, 3, 1, 2)
    for k in ([0] if scale in (2, 3) else [0, 2]):                                # the oracle's Upsample (hit_sir_pro.py:1024-1043)
        y = torch.nn.functional.pixel_shuffle(torch.nn.functional.conv2d(y, sd[f"upsample.{k}.weight"], sd[f"upsample.{k}.bias"], 1, 1),
                                              3 if scale == 3 else 2)
    want = (torch.nn.functional.conv2d(y, sd["conv_last.weight"], sd["conv_last.bias"], 1, 1) + oracle.mean).permute(0, 2, 3, 1)
    fp32_noise("pixelshuffle", sr.head_pixelshuffle(u0, sd, scale, sr.PIN)[0], want)
    ref, bound = sr.head_pixelshuffle(u0, sd, scale, sr.REF)
    sr.check_bound(f"pixelshuffle x{scale} sim", sr.head_pixelshuffle(u0, sd, scale, sr.SIM)[0], ref, bound)
    rejected("sub-pixel transposed", sr.head_pixelshuffle(u0, sd, scale, sr.SIM, {"ps_transposed"})[0], ref, bound)


@pytest.mark.parametrize("scale", [2, 3, 4])
def test_head_pixelshuffledirect(scale):
    _, oracle = build_pair((1, 1, 1), "pixelshuffledirect", scale, "stress", 31)
    sd = oracle.sd
    f = noise_map(2, 9, 11, 180, seed=10 + scale)
    want = (torch.nn.functional.pixel_shuffle(torch.nn.functional.conv2d(f.permute(0, 3, 1, 2), sd["upsample.0.weight"],
                                                                        sd["upsample.0.bias"], 1, 1), scale) + oracle.mean)
    fp32_noise("pixelshuffledirect", sr.head_direct(f, sd, scale, sr.PIN)[0], want.permute(0, 2, 3, 1))
    ref, bound = sr.head_direct(f, sd, scale, sr.REF)
    sr.check_bound(f"pixelshuffledirect x{scale} sim", sr.head_direct(f, sd, scale, sr.SIM)[0], ref, bound)
    rejected("sub-pixel transposed", sr.head_direct(f, sd, scale, sr.SIM, {"ps_transposed"})[0], ref, bound)


def test_head_none():
    _, oracle = build_pair((1, 1, 1), None, 4, "stress", 31)
    sd = oracle.sd
    f, x = noise_map(2, 9, 11, 180, seed=20), torch.rand(2, 9, 11, 3)
    want = x + torch.nn.functional.conv2d(f.permute(0, 3, 1, 2), sd["conv_last.weight"], sd["conv_last.bias"], 1, 1).permute(0, 2, 3, 1)
    fp32_noise("upsampler=None", sr.head_none(f, x, sd, sr.PIN)[0], want)
    ref, bound = sr.head_none(f, x, sd, sr.REF)
    sr.check_bound("upsampler=None sim", sr.head_none(f, x, sd, sr.SIM)[0], ref, bound)
    rejected("input not added", sr.head_none(f, torch.zeros_like(x), sd, sr.SIM)[0], ref, bound)


@pytest.mark.parametrize("p", ["layers.0.conv.", "conv_after_body."])
def test_resi_3conv(p):
    from oracle.hitsir_oracle import resi_conv
    _, oracle = build_pair((1, 1, 1), "nearest+conv", 4, "stress", 21, resi_connection="3conv")
    sd = oracle.sd
    x = noise_map(2, 9, 11, 180, seed=30)
    res = noise_map(2, 9, 11, 180, seed=31) if p.startswith("layers") else None
    want = resi_conv(x, sd, p) + (0 if res is None else res)
    fp32_noise("3conv", sr.resi_3conv(x, sd, p, sr.PIN, res)[0], want)
    ref, bound = sr.resi_3conv(x, sd, p, sr.REF, res)
    sr.check_bound("3conv sim", sr.resi_3conv(x, sd, p, sr.SIM, res)[0], ref, bound)
    rejected("taps transposed", sr.resi_3conv(x, sd, p, sr.SIM, res, {"taps_transposed"})[0], ref, bound)


# ---- casa gate ----------------------------------------------------------------------------------------------------------------
WINDOWS = (4, 8, 16, 32, 48, 64)


@pytest.mark.parametrize("j", range(6))
def test_casa_qkv(net, j):
    """Block input -> the gated, reflect-padded token map (tap `block0.j.qkv`).  At 33 x 37 every window size pads both axes, so
    the reflected strips carry pixels that count twice in the pools and the gate convs read mirrored statistics at the edge.
    Pools over the unpadded map are rejected at w = 4, 8, 16 and 48 only: at w = 32 and 64 they move no output element by more than
    about half its bound (the bound there is dominated by the bf16 ulp of the stored token), so that mutant is not checked there."""
    sd, taps = net
    P, x, win = sr.block_params(sd, 0, j), block_input(taps, j), WINDOWS[j]
    fp32_noise("qkv", sr.casa_qkv(x, P, win, sr.PIN)[0], taps[f"block0.{j}.qkv"])
    ref, bound = sr.casa_qkv(x, P, win, sr.REF)
    sr.check_bound(f"casa w={win} sim", sr.casa_qkv(x, P, win, sr.SIM)[0], ref, bound)
    for mut in ("halo_zero", "lrelu_slope") + (() if win in (32, 64) else ("pool_unpadded",)):
        rejected(mut, sr.casa_qkv(x, P, win, sr.SIM, {mut})[0], ref, bound)


def test_casa_qkv_large_mean(net):
    """The shifted case of the GPU test: block input + 256 on every channel, so the pooled means are large next to the gate."""
    sd, taps = net
    P, x = sr.block_params(sd, 0, 0), taps["embed"] + 256.0
    ref, bound = sr.casa_qkv(x, P, 4, sr.REF)
    sr.check_bound("casa sim, large mean", sr.casa_qkv(x, P, 4, sr.SIM)[0], ref, bound)


# ---- entry: mean shift + conv_first -------------------------------------------------------------------------------------------
def test_entry_multi_size(net):
    sd, taps = net
    x = synthetic_image(B, H, W, seed=4)
    fp32_noise("shallow", sr.entry(x, sd, sr.PIN)[0], taps["shallow"])
    ref, bound = sr.entry(x, sd, sr.REF)
    sr.check_bound("entry sim", sr.entry(x, sd, sr.SIM)[0], ref, bound)
    for mut in ("gate_no_residual", "mean_added"):
        rejected(mut, sr.entry(x, sd, sr.SIM, mut={mut})[0], ref, bound)


def saturating_entry(sd):
    """conv_x scaled by 8: x1 x_k reaches |z| ~ 20, where the gate's sigmoid saturates (ex2 over- and underflows towards 0 and inf)."""
    sd = dict(sd)
    sd["conv_first.conv_x.weight"] = sd["conv_first.conv_x.weight"] * 8.0
    return sd


def test_entry_saturated_gate(net):
    sd, _ = net
    sd = saturating_entry(sd)
    x = synthetic_image(B, H, W, seed=4)
    ref, bound = sr.entry(x, sd, sr.REF)
    sr.check_bound("entry sim, saturated gate", sr.entry(x, sd, sr.SIM)[0], ref, bound)
    rejected("gate_no_residual", sr.entry(x, sd, sr.SIM, mut={"gate_no_residual"})[0], ref, bound)


def test_entry_conv_first():
    _, oracle = build_pair((0, 0, 0), "nearest+conv", 4, "stress", 21)
    sd = oracle.sd
    x = synthetic_image(B, H, W, seed=4)
    taps = {}
    with torch.no_grad():
        oracle.forward(x, taps)
    fp32_noise("shallow", sr.entry(x, sd, sr.PIN, ms=False)[0], taps["shallow"])
    ref, bound = sr.entry(x, sd, sr.REF, ms=False)
    sr.check_bound("conv_first sim", sr.entry(x, sd, sr.SIM, ms=False)[0], ref, bound)
    rejected("mean_added", sr.entry(x, sd, sr.SIM, ms=False, mut={"mean_added"})[0], ref, bound)


# ---- fusion ------------------------------------------------------------------------------------------------------------------
def test_fusion(net):
    sd, taps = net
    cab, s = taps["conv_after_body"], taps["shallow"]
    fp32_noise("fused", sr.fusion(cab, s, sd, sr.PIN)[0], taps["fused"])
    ref, bound = sr.fusion(cab, s, sd, sr.REF)
    sr.check_bound("fusion sim", sr.fusion(cab, s, sd, sr.SIM)[0], ref, bound)
    for mut in ("swap", "sig_outside", "ch_h_not_transposed", "planes_swapped"):
        rejected(mut, sr.fusion(cab, s, sd, sr.SIM, {mut})[0], ref, bound)


# ---- window self-correlation --------------------------------------------------------------------------------------------------
def pooled_bias(sd, j):
    from oracle.hitsir_oracle import dynamic_pos_bias_table, pooled_rpe_bias
    win = WINDOWS[j]
    tbl = dynamic_pos_bias_table(sd, f"layers.0.residual_group.blocks.{j}.correlation.", (win, win))
    return pooled_rpe_bias(tbl, (win, win), (min(win, 8), min(win, 8)))


SCC_MUTANTS = ("no_bsl_vpt", "no_bsl_kp", "scale16", "inv_lb", "kgen_swapped", "no_ones", "bias_transposed", "bias_xy")
SCC_UNREJECTED = {16: ("no_bsl_vpt", "no_bsl_kp", "no_ones"), 32: ("no_bsl_kp", "no_ones"), 48: ("no_bsl_vpt", "no_bsl_kp", "no_ones"),
                  64: ("no_bsl_vpt", "no_bsl_kp", "no_ones")}


@pytest.mark.parametrize("j", range(6))
def test_scc(net, j):
    """Tap `block0.j.qkv` (the padded token map) + the pooled bias -> tap `block0.j.scc`; SIM is `scc_dense` for w = 4, 8 and
    `scc_umma` for w >= 16.  Mutants that do not apply to a kernel are skipped: "bias_transposed" needs the square L x L table of
    `scc_dense`, "bias_xy" is its `scc_umma` counterpart, and "inv_lb" is no bug at r = 1 (Lb = L).
    Not rejected at this shape (`SCC_UNREJECTED`): in `scc_umma` the bound is dominated by the bf16 rounding of G = Q^T T, a sum over
    L tokens carried through |Wk| / L and |V|, and of KP; spatial_linear.bias and the k-gen bias move the output by less than that at
    w = 16, 48, 64 (no_bsl_vpt, no_bsl_kp, no_ones; worst ratios 0.16 .. 1.0), and at w = 32 for no_bsl_kp (1.08, too close to 1 to
    count) and no_ones.  Each of them is rejected at w = 4 and 8, and no_bsl_vpt also at w = 32."""
    sd, taps = net
    P, win = sr.block_params(sd, 0, j), WINDOWS[j]
    bias = pooled_bias(sd, j)
    tok = taps[f"block0.{j}.qkv"]
    fp32_noise("scc", sr.scc(tok, bias, P, win, sr.PIN, (H, W))[0], taps[f"block0.{j}.scc"])
    tok = sr.bf(tok).float()
    ref, bound = sr.scc(tok, bias, P, win, sr.REF, (H, W))
    sr.check_bound(f"scc w={win} sim", sr.scc(tok, bias, P, win, sr.SIM, (H, W))[0], ref, bound)
    dense = win <= 8
    for mut in SCC_MUTANTS:
        if (mut == "bias_xy" and dense) or (mut in ("bias_transposed",) and not dense) or (mut == "inv_lb" and dense) \
                or mut in SCC_UNREJECTED.get(win, ()):
            continue
        rejected(mut, sr.scc(tok, bias, P, win, sr.SIM, (H, W), {mut})[0], ref, bound)
