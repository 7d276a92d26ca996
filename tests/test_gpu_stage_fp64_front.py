"""The window self-correlation, the casa gate, the entry and the fusion in isolation against an fp64 evaluation of their own
exact inputs (-m gpu).

Same method as tests/test_gpu_stage_fp64.py: each stage is fed the values its kernels read (a tap or an injection of one seeded
forward), its output tap is compared element by element with the a-priori bound of tests/stage_ref.py (`scc`, `casa_qkv`,
`entry`, `fusion`), and each check prints its worst |got - ref| / bound.  tests/test_stage_ref.py shows on the CPU that the simulated kernels
pass these bounds and that plausible mutants of them do not.

Two shapes, chosen for the kernels' edge cases:
  trunk: B = 2, 98 x 146 -- w = 4 gives 925 windows per image and w = 8 gives 247, so one 128-token `scc_dense` tile holds windows of
         both images and the last tile is partial; w = 48 and 64 pad 46 columns and run `scc_umma`'s streaming mode (18 and 32 token
         tiles per window, phase B walked backwards); w = 16 runs its two-tile mode.  The casa statistics come from `sca_stats`
         (block 0, injections) or from the previous `ffn_tail`'s statistics warp (blocks 1..5);
  small: B = 1, 37 x 53 -- at w = 8, 35 windows make 18 `scc_dense` tiles, fewer than the SMs, so the CTA of the last tile gets only
         that partial tile: the rows of its absent windows are never loaded and are multiplied by the exact zeros of the masked P
         operands (a stale NaN there would show as a non-finite output); at w = 4, 140 windows leave a partial last tile too."""
import pytest
import torch

from oracle.weights import synthetic_image
from tests import stage_ref as sr
from tests.helpers import build_pair
from tests.test_gpu_stage_fp64 import DEV, C, tap

pytestmark = pytest.mark.gpu
SHAPES = {"trunk": (2, 98, 146), "small": (1, 37, 53)}
WINDOWS = (4, 8, 16, 32, 48, 64)


def make_model(flags=(1, 1, 1), edit=None, **extra):
    model, oracle = build_pair(flags, "nearest+conv", 4, "stress", 21, edit=edit, **extra)
    return model.to(DEV), oracle.sd


@pytest.fixture(scope="module")
def trunk():
    model, sd = make_model()
    B, H, W = SHAPES["trunk"]
    return model, sd, synthetic_image(B, H, W, seed=4).to(DEV)


@pytest.fixture(scope="module")
def small():
    model, sd = make_model()
    B, H, W = SHAPES["small"]
    return model, sd, synthetic_image(B, H, W, seed=6).to(DEV)


def padded(n, w):
    return (n + w - 1) // w * w


# ---- window self-correlation ------------------------------------------------------------------------------------------------
def check_scc(model, sd, x, j, name):
    """Tap `block0.j.qkv` (the token map the kernel reads) and tap `block0.j.scc` of the same seeded forward, with the bias table the
    library precomputed."""
    B, H, W = x.shape[0], x.shape[2], x.shape[3]
    tok = qkv_tap(model, x, j)
    got = tap(model, x, f"block0.{j}.scc", (B, H, W, C))
    bias = model.bias_table(DEV, 0, j).cpu()
    ref, bound = sr.scc(tok, bias, sr.block_params(sd, 0, j), WINDOWS[j], sr.REF, (H, W))
    sr.check_bound(f"scc block0.{j} (w = {WINDOWS[j]}) {name}", got, ref, bound)


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("j", range(6))
def test_scc(request, shape, j):
    model, sd, x = request.getfixturevalue(shape)
    check_scc(model, sd, x, j, shape)


@pytest.mark.parametrize("j", [1, 4])
def test_scc_common_mode(j):
    """casa off, block input injected with +64 on every channel: G, TPT and KP (and the scores of `scc_dense`) are then much larger
    than the output, so the bf16 rounding of those intermediates, not the output's, sets the bound (w = 8: `scc_dense`, w = 48:
    `scc_umma` streaming)."""
    model, sd = make_model((1, 0, 1))
    B, H, W = SHAPES["trunk"]
    x = synthetic_image(B, H, W, seed=4).to(DEV)
    src = tap(model, x, "embed", (B, H, W, C)) + 64.0
    model.set_inject(DEV, f"block0.{j}.in", src.reshape(-1, C).to(DEV))
    try:
        check_scc(model, sd, x, j, "casa off, +64")
    finally:
        model.set_inject(DEV, None)


@pytest.mark.parametrize("base,j", [(4, 1), (4, 2), (2, 0), (2, 1)])
def test_scc_pooled_base(base, j):
    """base_win_size below 8, windows 4..64 as in the pro model: the w = 4 / 8 windows pool inside their one token tile and run
    `scc_umma`'s resident mode (base 4: w = 8 at r = 2; base 2: w = 4 at r = 2, w = 8 at r = 4); base 4, w = 16 runs the two-tile
    mode over 16 pooled cells (one cell k-step)."""
    model, sd = make_model(base_win_size=[base, base], hier_win_ratios=[w / base for w in WINDOWS])
    B, H, W = SHAPES["trunk"]
    check_scc(model, sd, synthetic_image(B, H, W, seed=4).to(DEV), j, f"base_win_size {base}")


# ---- casa gate --------------------------------------------------------------------------------------------------------------
def qkv_tap(model, x, j):
    B, H, W = x.shape[0], x.shape[2], x.shape[3]
    w = WINDOWS[j]
    return tap(model, x, f"block0.{j}.qkv", (B, padded(H, w), padded(W, w), C))


@pytest.mark.parametrize("j", range(6))
def test_casa_from_stream(trunk, j):
    """Block input (tap `embed` for j = 0, else tap `block0.{j-1}`) -> tap `block0.j.qkv`.  For j >= 1 the pools are the ones
    `ffn_tail`'s statistics warp produced, weighted by the reflect multiplicity of this block's window padding."""
    model, sd, x = trunk
    B, H, W = SHAPES["trunk"]
    xin = tap(model, x, "embed" if j == 0 else f"block0.{j - 1}", (B, H, W, C))
    got = qkv_tap(model, x, j)
    ref, bound = sr.casa_qkv(xin, sr.block_params(sd, 0, j), WINDOWS[j], sr.REF)
    sr.check_bound(f"casa block0.{j} (w = {WINDOWS[j]})", got, ref, bound)


@pytest.mark.parametrize("j,shift", [(j, 0.0) for j in range(6)] + [(0, 256.0)])
def test_casa_injected(trunk, j, shift):
    """Injected block input -> tap `block0.j.qkv`: the injection discards the delivered statistics, so this path runs `sca_stats`.
    shift = 256 adds 256 to every channel of the injected stream: the pooled means are then large next to the gate."""
    model, sd, x = trunk
    B, H, W = SHAPES["trunk"]
    src = tap(model, x, "embed", (B, H, W, C)) + shift
    model.set_inject(DEV, f"block0.{j}.in", src.reshape(-1, C).to(DEV))
    try:
        got = qkv_tap(model, x, j)
    finally:
        model.set_inject(DEV, None)
    ref, bound = sr.casa_qkv(src, sr.block_params(sd, 0, j), WINDOWS[j], sr.REF)
    sr.check_bound(f"casa block0.{j} injected (+{shift:g})", got, ref, bound)


# ---- entry ------------------------------------------------------------------------------------------------------------------
def saturating_gate(sd):
    """conv_x scaled by 8: x1 x_k reaches |z| ~ 20, where the gate's sigmoid saturates."""
    sd["conv_first.conv_x.weight"] *= 8.0


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("flags,planted", [((1, 1, 1), False), ((0, 0, 0), False), ((1, 1, 1), True)])
def test_entry(shape, flags, planted):
    """The image -> tap `shallow` (fp32): `entry_im2col` + the conv_first GEMM (EPI_MSGATE + conv_first.conv_last with the
    multi-size extractor, a plain 3 x 3 conv without it)."""
    model, sd = make_model(flags, saturating_gate if planted else None)
    B, H, W = SHAPES[shape]
    x = synthetic_image(B, H, W, seed=5)
    got = tap(model, x.to(DEV), "shallow", (B, H, W, C))
    ref, bound = sr.entry(x, sd, sr.REF, ms=bool(flags[0]))
    sr.check_bound(f"entry {flags} {shape}" + (" saturated gate" if planted else ""), got, ref, bound)


# ---- fusion -----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", SHAPES)
def test_fusion(request, shape):
    """Taps `conv_after_body` (first) and `shallow` (second) -> the fp32 tap `fused` that `fusion_combine` writes."""
    model, sd, x = request.getfixturevalue(shape)
    B, H, W = SHAPES[shape]
    cab = tap(model, x, "conv_after_body", (B, H, W, C))
    shallow = tap(model, x, "shallow", (B, H, W, C))
    got = tap(model, x, "fused", (B, H, W, C))
    ref, bound = sr.fusion(cab, shallow, sd, sr.REF)
    sr.check_bound(f"fusion {shape}", got, ref, bound)
