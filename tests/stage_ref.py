"""fp64 references of single CUDA stages and element-wise error bounds derived from each stage's arithmetic -- TEST INFRASTRUCTURE.

A stage is fed the exact values its kernel consumes (a tap or an injection of a deterministic forward), so the only error left in its
output is the stage's own arithmetic.  Every stage function here evaluates one stage under an `Arith`:

* `REF`: float64 with the operands the kernel reads -- bf16(w) for every packed weight and every bf16 activation operand, fp32 biases,
  LayerNorm parameters and scalars -- and no intermediate rounding.  Its output is what the tests compare the kernel with.
* `SIM`: the simulated kernel: float32, the same bf16 operands, and bf16 rounding at the intermediate sites the kernel has (and of its
  output where the kernel stores bf16).  `tests/test_stage_ref.py` shows it passes the bound and that plausible mutants of it do not.
* `PIN`: float64 with the oracle's own fp32 operands, which pins each stage function to the oracle's taps (`oracle/hitsir_oracle.py`).

The a-priori bound of an output element is

    |got - ref| <= K * 2^-22 * M_acc  +  sum over bf16 rounding sites of 2^-8 * M_site  +  ulp_out(ref)

where M_acc is the magnitude pass (the same contraction evaluated on |operands|) of a reduction of length K (2^-22 instead of the fp32
unit roundoff 2^-24 covers the tensor core's non-IEEE accumulation), M_site is the magnitude of an intermediate the kernel rounds to bf16,
carried to the output by the magnitude pass of what follows it, and ulp_out is one ulp of the stored output type.  LayerNorm and GELU
propagate the bound of their input as derived at `ln_bound` and `gelu_bound`.  No constant here is a measurement of the kernel it judges.
"""
from __future__ import annotations

from dataclasses import dataclass

import torch
import torch.nn.functional as F

from tests.test_subpixel_identity import phase_filter, subpixel_conv

U32 = 2.0 ** -24          # fp32 unit roundoff (one rounded add, multiply or store)
UACC = 2.0 ** -22         # per term of an fp32 reduction on the tensor core or in a reduction tree
UBF = 2.0 ** -8           # one intermediate bf16 rounding, relative
GELU_LIP = 1.13           # max |GELU'(x)| = 1.1289 (x = sqrt(2))
RGB_MEAN = (0.485, 0.456, 0.4060)
NHWC = ("image", "y", "x", "channel")


def bf(t: torch.Tensor) -> torch.Tensor:
    """Round to bf16 the way the kernels do (from fp32, round to nearest even); returns float64."""
    return t.float().to(torch.bfloat16).double()


def ulp(ref: torch.Tensor, bf16: bool) -> torch.Tensor:
    """One ulp of the output type at |ref| (the stored value is within half of it of the exact fp32 value)."""
    m = 7 if bf16 else 23
    _, e = torch.frexp(ref.double().abs().clamp_min(2.0 ** -126))
    return torch.ldexp(torch.ones_like(ref, dtype=torch.float64), e - 1 - m)


def gelu_fit(x: torch.Tensor) -> torch.Tensor:
    """|gelu2(x) - GELU_erf(x)|.  gelu2 (common.cuh) is x/2 + x/2 * tanh(w) with w the quintic of DESIGN.md 3.1: the fit of the
    logistic to the normal CDF is within 1.6e-5 * max(|x|, 1), and PTX documents tanh.approx.f32 to a maximum relative error of
    2^-10.987, which x/2 * tanh(w) carries to 2^-11.987 * |x|."""
    a = x.abs()
    return 1.6e-5 * a.clamp_min(1.0) + 2.0 ** -11.987 * a


@dataclass(frozen=True)
class Arith:
    dtype: torch.dtype
    bf16_operands: bool
    bf16_sites: bool

    def op(self, t):
        """An operand the kernel reads as bf16 (packed weight, bf16 activation)."""
        return (bf(t) if self.bf16_operands else t.double()).to(self.dtype)

    def f32(self, t):
        """An operand the kernel reads in fp32 (bias, LayerNorm parameter, fp32 residual stream)."""
        return t.to(self.dtype)

    def site(self, t):
        """An intermediate the kernel rounds to bf16."""
        return bf(t).to(self.dtype) if self.bf16_sites else t

    def out(self, t, bf16: bool):
        """The stored output: bf16 outputs are rounded in the simulated kernel; the reference stays exact (ulp_out covers it)."""
        return bf(t).to(self.dtype) if (bf16 and self.bf16_sites) else t


REF = Arith(torch.float64, True, False)
SIM = Arith(torch.float32, True, True)
PIN = Arith(torch.float64, False, False)


# --------------------------------------------------------------------------------------------------------------------------------
# bound pieces
# --------------------------------------------------------------------------------------------------------------------------------
def ln_bound(pre: torch.Tensor, e_pre: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float = 1e-5) -> torch.Tensor:
    """Bound of |LN_kernel(pre~) - LN(pre)| per element, where pre is the exact pre-norm row (C values) and pre~ the kernel's, with
    |pre~ - pre| <= e_pre.  The kernels compute the mean, then the centred second moment (two-pass in `ln_rows`, per-slice (mean, M2)
    merged with Chan's update in the GEMM and FFN-tail epilogues -- both sum the same centred squares), then rsqrt:

        mean:   e_mu  = mean(e_pre) + C * 2^-22 * mean|pre|                 (input error + reduction)
        centre: e_d   = e_pre + e_mu + 2^-24 |d|,        d = pre - mean
        var:    e_var = mean(2 |d| e_d + e_d^2) + C * 2^-22 * var           (squares of perturbed d + reduction)
        rstd:   rho = e_var / (var + eps);  |r~/r - 1| <= rho / (2 (1 - rho)^1.5) + 2^-21     (rsqrt approximation: 2 ulp)
        out:    e_y   = |g| r (e_d (1 + rel_r) + |d| rel_r) + 3 * 2^-24 (|d| r |g| + |b|)

    The last line is the first-order expansion of (d + e_d) r (1 + rel_r) g + b; its second-order term is the e_d rel_r product."""
    C = pre.shape[-1]
    mu = pre.mean(-1, keepdim=True)
    d = pre - mu
    var = (d * d).mean(-1, keepdim=True)
    e_mu = e_pre.mean(-1, keepdim=True) + C * UACC * pre.abs().mean(-1, keepdim=True)
    e_d = e_pre + e_mu + U32 * d.abs()
    e_var = (2 * d.abs() * e_d + e_d * e_d).mean(-1, keepdim=True) + C * UACC * var
    rho = e_var / (var + eps)
    rel_r = torch.where(rho < 0.5, rho / (2 * (1 - rho.clamp(max=0.5)) ** 1.5) + 2.0 ** -21, torch.full_like(rho, float("inf")))
    r = 1.0 / torch.sqrt(var + eps)
    g, b = gamma.double().abs(), beta.double().abs()
    e = g * r * (e_d * (1 + rel_r) + d.abs() * rel_r) + 3 * U32 * (d.abs() * r * g + b)
    return torch.nan_to_num(e, nan=float("inf"))


def gelu_bound(pre: torch.Tensor, e_pre: torch.Tensor) -> torch.Tensor:
    """|gelu2(pre~) - GELU(pre)| <= max|GELU'| e_pre + fit error (GELU is 1.13-Lipschitz)."""
    return GELU_LIP * e_pre + gelu_fit(pre)


def block_params(sd, i: int, j: int) -> dict:
    """The parameters of block i.j keyed as the stage functions use them ("proj.weight", "norm1.weight", "fc1.weight", ...)."""
    p = f"layers.{i}.residual_group.blocks.{j}."
    out = {}
    for k, v in sd.items():
        if k.startswith(p):
            k = k[len(p):]
            for sub in ("correlation.", "mlp."):
                k = k[len(sub):] if k.startswith(sub) else k
            out[k] = v
    return out


def _lin(a, w, b=None):
    y = a @ w.t()
    return y if b is None else y + b


def _conv(x, w, b=None, pad=1, groups=1):
    """Conv2d on NHWC."""
    return F.conv2d(x.permute(0, 3, 1, 2), w, b, 1, pad, 1, groups).permute(0, 2, 3, 1)


def _nnz_k(w: torch.Tensor) -> int:
    """Reduction length of a contraction: the largest number of non-zero weights of one output, plus the bias.  Adding an exact zero
    product is exact, so planted sparse weights get the (tighter, still rigorous) bound of their real reduction length."""
    return int((w.reshape(w.shape[0], -1) != 0).sum(1).max().item()) + 1


# --------------------------------------------------------------------------------------------------------------------------------
# stages: each returns (out, bound); the bound is computed in float64 from the REF operands whatever `ar` is
# --------------------------------------------------------------------------------------------------------------------------------
def layer_norm(x, g, b, mut=()):
    eps = 1e-6 if "ln_eps" in mut else 1e-5
    mu = x.mean(-1, keepdim=True)
    if "ln_onepass" in mut:
        var = (x * x).mean(-1, keepdim=True) - mu * mu
    else:
        var = ((x - mu) ** 2).mean(-1, keepdim=True)
    return (x - mu) / torch.sqrt(var + eps) * g + b


def ln_rows(x, g, b, ar: Arith, bf16_out: bool, mut=()):
    """`ln_rows` (patch_embed norm :975-983 with fp32 output, final norm :1299 with bf16 output): reads the fp32 stream exactly.
    Rounding sites: none inside; the output (bf16 for the final norm)."""
    out = ar.out(layer_norm(ar.f32(x), ar.f32(g), ar.f32(b), mut), bf16_out)
    x64 = x.double()
    ref = layer_norm(x64, g.double(), b.double())
    return out, ln_bound(x64, torch.zeros_like(x64), g, b) + ulp(ref, bf16_out)


def proj_norm1(scc, xin, P, ar: Arith, mut=()):
    """proj + norm1 + residual (:597, :700-703), the TMA LayerNorm epilogue of `umma_gemm_tma_kernel<192>`: A = the bf16 SCC output
    (exact), fp32 bias, LayerNorm statistics of the fp32 accumulator row, + the fp32 stream.  K = 180 (+ bias).
    Rounding sites: none; the fp32 output (ulp) and the residual add (2^-24 |out|)."""
    w, b = P["proj.weight"], P["proj.bias"]
    res = ar.op(xin) if "res_bf16" in mut else ar.f32(xin)
    pre = _lin(ar.op(scc), ar.op(w), ar.f32(b))
    out = res + layer_norm(pre, ar.f32(P["norm1.weight"]), ar.f32(P["norm1.bias"]), mut)
    a, wq = bf(scc), bf(w)
    pre64 = _lin(a, wq, b.double())
    e_pre = _nnz_k(w) * UACC * _lin(a.abs(), wq.abs(), b.double().abs())
    ref = xin.double() + layer_norm(pre64, P["norm1.weight"].double(), P["norm1.bias"].double())
    return out, ln_bound(pre64, e_pre, P["norm1.weight"], P["norm1.bias"]) + U32 * ref.abs() + ulp(ref, False)


def fc1_gelu(attn, P, ar: Arith, mut=()):
    """fc1 + GELU (:39-41), the activation epilogue of `umma_gemm_tma_kernel<192>` with resident weights: A = bf16 shadow of the
    stream, fp32 bias, `gelu2`, bf16 store.  K = 180 (+ bias).  Rounding sites: none inside; the bf16 output (ulp).
    Returns (out, bound, pre) -- `pre`, the exact pre-activation, is the x of the binned-mean check."""
    w, b = P["fc1.weight"], P["fc1.bias"]
    pre = _lin(ar.op(attn), ar.op(w), ar.f32(b))
    if "gelu_sigmoid" in mut:
        out = ar.out(pre * torch.sigmoid(1.702 * pre), True)
    else:
        out = ar.out(F.gelu(pre), True)
    a, wq = bf(attn), bf(w)
    pre64 = _lin(a, wq, b.double())
    e_pre = _nnz_k(w) * UACC * _lin(a.abs(), wq.abs(), b.double().abs())
    ref = F.gelu(pre64)
    return out, gelu_bound(pre64, e_pre) + ulp(ref, True), pre64


def ffn_tail(h1, attn, P, ar: Arith, mut=()):
    """`ffn_tail_kernel` (:42-46, :704): dwconv 5x5 on mma.sync (bf16 taps, fp32 bias, K = 25 + 1) + GELU (`gelu2`) + input -> h2,
    rounded to bf16 as the A operand of fc2 (site 1); fc2 (K = 360 + 1) into TMEM, LayerNorm epilogue + the fp32 stream.
    Bound: e_dw = 26 * 2^-22 * M_dw, e_h2 = 1.13 e_dw + fit + 2^-8 (|h1| + |GELU(dw)|) (site 1), e_pre2 = |W2| e_h2 +
    361 * 2^-22 * M_fc2, then `ln_bound`, + 2^-24 |out| for the residual add and one fp32 ulp."""
    wd, bd = P["dwconv.depthwise_conv.0.weight"], P["dwconv.depthwise_conv.0.bias"]
    w2, b2 = P["fc2.weight"], P["fc2.bias"]
    C = wd.shape[0]
    wdm = wd.transpose(-1, -2) if "dw_transposed" in mut else wd
    x = ar.op(h1)
    dw = _conv(x, ar.op(wdm), ar.f32(bd), 2, C)
    h2 = ar.site(x + F.gelu(dw))
    pre2 = _lin(h2, ar.op(w2), ar.f32(b2))
    res = ar.op(attn) if "res_bf16" in mut else ar.f32(attn)
    out = res + layer_norm(pre2, ar.f32(P["norm2.weight"]), ar.f32(P["norm2.bias"]), mut)
    x64, wd64, w264 = bf(h1), bf(wd), bf(w2)
    dw64 = _conv(x64, wd64, bd.double(), 2, C)
    e_dw = 26 * UACC * _conv(x64.abs(), wd64.abs(), bd.double().abs(), 2, C)
    g64 = F.gelu(dw64)
    h264 = x64 + g64
    e_h2 = gelu_bound(dw64, e_dw) + UBF * (x64.abs() + g64.abs())
    pre264 = _lin(h264, w264, b2.double())
    e_pre2 = _lin(e_h2, w264.abs()) + _nnz_k(w2) * UACC * _lin(h264.abs(), w264.abs(), b2.double().abs())
    ref = attn.double() + layer_norm(pre264, P["norm2.weight"].double(), P["norm2.bias"].double())
    return out, ln_bound(pre264, e_pre2, P["norm2.weight"], P["norm2.bias"]) + U32 * ref.abs() + ulp(ref, False)


def conv3(x, w, b, ar: Arith, res=None, slope=None, bf16_out=False, mut=()):
    """A 3x3 conv on `umma_gemm_tma_kernel` / `conv3_c64_kernel` (implicit GEMM, zero padding by TMA OOB fill): A = bf16 NHWC map,
    bf16 weights, fp32 bias [+ fp32 residual] [LeakyReLU(slope)], fp32 or bf16 store.  K = 9 * Ci (+ bias).  Rounding sites: none
    inside; the output (ulp), the residual add (2^-24 |out|).  LeakyReLU is 1-Lipschitz."""
    y = _conv(ar.op(x), ar.op(w), ar.f32(b))
    if res is not None:
        y = y + ar.f32(res)
    if slope is not None:
        y = F.leaky_relu(y, (0.2 if slope == 0.01 else 0.01) if "lrelu_slope" in mut else slope)
    out = ar.out(y, bf16_out)
    x64, w64 = bf(x), bf(w)
    ref = _conv(x64, w64, b.double())
    e = _nnz_k(w) * UACC * _conv(x64.abs(), w64.abs(), b.double().abs())
    if res is not None:
        ref = ref + res.double()
        e = e + U32 * ref.abs()
    if slope is not None:
        ref = F.leaky_relu(ref, slope)
    return out, e + ulp(ref, bf16_out)


def phase_filter_bf16(w, a, bb, dyi, dxi):
    """The phase filter as `pack_subpixel_kernel` stores it: the fp32 tap sum rounded once to bf16."""
    return bf(phase_filter(w.float(), a, bb, dyi, dxi))


def conv_up(x, w, b, ar: Arith, mut=()):
    """interpolate(x2, nearest) + conv3x3 64 -> 64 + LeakyReLU(0.2) (:1331-1332) as `conv3_c64_up_kernel`: four 2x2 sub-pixel convs of
    the LR map with the bf16 phase filters (K = 4 * 64 + bias per output), bf16 store.  Rounding sites: none inside (the filters are
    operands); the bf16 output (ulp).  Output NHWC (B, 2H, 2W, 64)."""
    base = phase_filter_bf16 if ar.bf16_operands else (lambda w_, *s: phase_filter(w_.double(), *s))
    swap = "phase_swap" in mut

    def filt(w_, a, bb, dyi, dxi):
        return (base(w_, bb, a, dyi, dxi) if swap else base(w_, a, bb, dyi, dxi)).to(ar.dtype)
    y = F.leaky_relu(subpixel_conv(ar.op(x).permute(0, 3, 1, 2), w, ar.f32(b), filt), 0.2)
    out = ar.out(y.permute(0, 2, 3, 1), True)
    x64 = bf(x).permute(0, 3, 1, 2)
    ref = F.leaky_relu(subpixel_conv(x64, w, b.double(), phase_filter_bf16), 0.2).permute(0, 2, 3, 1)
    mag = subpixel_conv(x64.abs(), w, b.double().abs(), lambda *s: phase_filter_bf16(*s).abs()).permute(0, 2, 3, 1)
    return out, (4 * w.shape[1] + 1) * UACC * mag + ulp(ref, True)


def conv_last(x, w, b, ar: Arith, img_range=1.0, mean=RGB_MEAN):
    """conv_last 64 -> 3 (+ mean, NCHW fp32, :1334, :1342) as `conv_last_fold_kernel`: per input pixel one contraction by all nine taps
    (K = 64, fp32 products in shared memory), the nine shifted partials added in fp32: K = 9 * 64 + bias terms of one reduction.
    Rounding sites: none; the fp32 output and the mean add (2 ulp).  Returns NHWC (B, H, W, 3)."""
    m = torch.tensor(mean[:w.shape[0]], dtype=ar.dtype)
    out = _conv(ar.op(x), ar.op(w), ar.f32(b)) / img_range + m
    x64, w64 = bf(x), bf(w)
    ref = _conv(x64, w64, b.double()) / img_range + m.double()
    e = _nnz_k(w) * UACC * _conv(x64.abs(), w64.abs(), b.double().abs()) / img_range
    return out, e + 2 * ulp(ref, False)


def pixel_shuffle(x, s: int, mut=()):
    """nn.PixelShuffle(s) on NHWC: channel c * s^2 + i * s + j goes to sub-pixel (i, j) of channel c.  Mutant "ps_transposed" swaps
    i and j."""
    xn = x.permute(0, 3, 1, 2)
    if "ps_transposed" in mut:
        B, C, H, W = xn.shape
        xn = xn.reshape(B, C // (s * s), s, s, H, W).transpose(2, 3).reshape(B, C, H, W)
    return F.pixel_shuffle(xn, s).permute(0, 2, 3, 1)


def _site(e_pre, v):
    """Error after storing an intermediate as bf16: the computed value v~ has |v~ - v| <= e_pre (v the exact value), and rounding to
    nearest adds at most half an ulp, <= 2^-8 |v~| <= 2^-8 (|v| + e_pre)."""
    return e_pre + UBF * (v.abs() + e_pre)


def head_pixelshuffle(u0, sd, s: int, ar: Arith, mut=(), img_range=1.0, mean=RGB_MEAN):
    """'pixelshuffle' head after conv_before_upsample (:1313-1319): Upsample = [conv3 64 -> 4*64 + PixelShuffle(2)] x log2(s) or
    [conv3 64 -> 9*64 + PixelShuffle(3)], each a `umma_gemm` conv with the EPI_SHUFFLE_BF16 direct-store epilogue (K = 576 + bias,
    bf16 store = rounding site 1 and, for x4, 2), then conv_last 64 -> 3 (+ mean, NCHW fp32, K = 576 + bias).  Input: the bf16 map
    `conv_before_upsample`.  Bound: per Upsample stage e = |W| * e_in + 577 * 2^-22 * M, then the site (`_site`); conv_last carries e
    through |W_last| and adds its own reduction term and 2 fp32 ulps (the mean add).  Returns NHWC (B, sH, sW, 3)."""
    r = 3 if s == 3 else 2
    y, y64 = ar.op(u0), bf(u0)
    e = torch.zeros_like(y64)
    for k in ([0] if s in (2, 3) else [0, 2]):
        w, b = sd[f"upsample.{k}.weight"], sd[f"upsample.{k}.bias"]
        y = ar.site(pixel_shuffle(_conv(y, ar.op(w), ar.f32(b)), r, mut))
        w64 = bf(w)
        m = _conv(y64.abs() + e, w64.abs(), b.double().abs())
        ez = _conv(e, w64.abs()) + _nnz_k(w) * UACC * m
        y64 = pixel_shuffle(_conv(y64, w64, b.double()), r)
        e = _site(pixel_shuffle(ez, r), y64)
    wl, bl = sd["conv_last.weight"], sd["conv_last.bias"]
    mv = torch.tensor(mean[:wl.shape[0]], dtype=torch.float64)
    out = _conv(y, ar.op(wl), ar.f32(bl)) / img_range + mv.to(ar.dtype)
    wl64 = bf(wl)
    ref = _conv(y64, wl64, bl.double()) / img_range + mv
    bound = (_conv(e, wl64.abs()) + _nnz_k(wl) * UACC * _conv(y64.abs() + e, wl64.abs(), bl.double().abs())) / img_range
    return out, bound + 2 * ulp(ref, False)


def head_direct(f, sd, s: int, ar: Arith, mut=(), img_range=1.0, mean=RGB_MEAN):
    """'pixelshuffledirect' (:1320-1325): conv3 180 -> 3 s^2 on the bf16 fused map with the EPI_SHUFFLE_NCHW direct-store epilogue
    (PixelShuffle(s), / img_range + mean, fp32 NCHW).  K = 1620 + bias; no rounding site; 2 fp32 ulps (the mean add).  NHWC out."""
    w, b = sd["upsample.0.weight"], sd["upsample.0.bias"]
    mv = torch.tensor(mean[:w.shape[0] // (s * s)], dtype=torch.float64)
    out = pixel_shuffle(_conv(ar.op(f), ar.op(w), ar.f32(b)), s, mut) / img_range + mv.to(ar.dtype)
    x64, w64 = bf(f), bf(w)
    ref = pixel_shuffle(_conv(x64, w64, b.double()), s) / img_range + mv
    e = pixel_shuffle(_nnz_k(w) * UACC * _conv(x64.abs(), w64.abs(), b.double().abs()), s) / img_range
    return out, e + 2 * ulp(ref, False)


def head_none(f, x_img, sd, ar: Arith, img_range=1.0):
    """upsampler=None (:1335-1342): y = x + conv_last(fused) / img_range, conv3 180 -> 3 on the bf16 fused map, the fp32 input image
    added in the epilogue (`res_img`).  K = 1620 + bias; no rounding site; 2 fp32 ulps.  x_img NHWC; NHWC out."""
    w, b = sd["conv_last.weight"], sd["conv_last.bias"]
    out = ar.f32(x_img) + _conv(ar.op(f), ar.op(w), ar.f32(b)) / img_range
    x64, w64 = bf(f), bf(w)
    ref = x_img.double() + _conv(x64, w64, b.double()) / img_range
    e = _nnz_k(w) * UACC * _conv(x64.abs(), w64.abs(), b.double().abs()) / img_range
    return out, e + 2 * ulp(ref, False)


def resi_3conv(x, sd, p: str, ar: Arith, res=None, mut=()):
    """resi_connection='3conv' (:913-918, :1224-1231) as engine.cu `resi_3conv`: t1 = LReLU0.2(conv3 180 -> 45) stored bf16 (site 1,
    K = 1620 + bias), t2 = LReLU0.2(conv1x1 45 -> 45) stored bf16 (site 2, K = 45 + bias), out = conv3 45 -> 180 (K = 405 + bias)
    [+ fp32 residual], fp32 store.  Input: the bf16 map.  Bound: each stage carries the previous error through |W| and adds its
    reduction term; each site adds 2^-8 (|t| + e) (`_site`); LeakyReLU is 1-Lipschitz; + 2^-24 |out| for the residual and one ulp."""
    wa, ba, wb, bb, wc, bc = (sd[p + k] for k in ("0.weight", "0.bias", "2.weight", "2.bias", "4.weight", "4.bias"))
    if "taps_transposed" in mut:
        wa = wa.transpose(-1, -2)
    t = ar.site(F.leaky_relu(_conv(ar.op(x), ar.op(wa), ar.f32(ba)), 0.2))
    t = ar.site(F.leaky_relu(_conv(t, ar.op(wb), ar.f32(bb), 0), 0.2))
    out = _conv(t, ar.op(wc), ar.f32(bc))
    t64 = bf(x)
    e = torch.zeros_like(t64)
    for w, b, pad in ((sd[p + "0.weight"], ba, 1), (wb, bb, 0)):
        w64 = bf(w)
        m = _conv(t64.abs() + e, w64.abs(), b.double().abs(), pad)
        ez = _conv(e, w64.abs(), None, pad) + _nnz_k(w) * UACC * m
        t64 = F.leaky_relu(_conv(t64, w64, b.double(), pad), 0.2)
        e = _site(ez, t64)
    wc64 = bf(wc)
    ref = _conv(t64, wc64, bc.double())
    bound = _conv(e, wc64.abs()) + _nnz_k(wc) * UACC * _conv(t64.abs() + e, wc64.abs(), bc.double().abs())
    if res is not None:
        out = out + ar.f32(res)
        ref = ref + res.double()
        bound = bound + U32 * ref.abs()
    return out, bound + ulp(ref, False)


# --------------------------------------------------------------------------------------------------------------------------------
# assertions
# --------------------------------------------------------------------------------------------------------------------------------
def check_bound(name: str, got: torch.Tensor, ref: torch.Tensor, bound: torch.Tensor, dims=NHWC) -> float:
    """Assert |got - ref| <= bound element by element.  Returns the worst ratio |got - ref| / bound; a failure names the worst element
    by `dims` (image, y, x, channel for NHWC maps)."""
    got, ref = got.double(), ref.double()
    assert got.shape == ref.shape == bound.shape, (name, got.shape, ref.shape, bound.shape)
    bad = ~torch.isfinite(got)
    if bad.any():
        i = [int(v) for v in torch.nonzero(bad)[0]]
        raise AssertionError(f"{name}: non-finite output at {dict(zip(dims, i))}")
    ratio = (got - ref).abs() / bound
    flat = int(torch.argmax(ratio))
    idx = [int(v) for v in torch.unravel_index(torch.tensor(flat), ratio.shape)]
    worst = ratio.reshape(-1)[flat].item()
    where = ", ".join(f"{k} {v}" for k, v in zip(dims, idx))
    msg = (f"{name}: worst |got - ref| / bound = {worst:.3g} at {where}: got {got.reshape(-1)[flat].item():.9g}, "
           f"ref {ref.reshape(-1)[flat].item():.9g}, bound {bound.reshape(-1)[flat].item():.3g}; "
           f"{int((ratio > 1).sum())} of {ratio.numel()} elements out of bound")
    print(msg)
    assert worst <= 1.0, msg
    return worst


def check_binned_mean(name: str, got: torch.Tensor, ref: torch.Tensor, x: torch.Tensor, width: float = 0.25, min_count: int = 256,
                      z: float = 6.0, x_max: float = 12.0, covers: float = 0.0) -> float:
    """Systematic error of an output-only nonlinearity: in every bin of width `width` of x (the exact pre-activation) with at least
    `min_count` elements and |x| <= x_max, the mean of (got - ref) must be within the fit error bound at the bin's largest |x| plus z
    standard errors of the mean (rounding of the stored value is unbiased and averages out; a wrong formula does not).  Equal x values
    round alike, so the standard error counts distinct x values only.  Some checked bin must lie at |x| >= `covers`.  Returns the
    worst ratio."""
    x, d = x.double().reshape(-1), (got.double() - ref.double()).reshape(-1)
    k = torch.floor(x / width).long()
    worst, where, reach = 0.0, None, 0.0
    for key in torch.unique(k).tolist():
        sel = k == key
        n = int(sel.sum())
        if n < min_count or max(abs(key * width), abs((key + 1) * width)) > x_max:
            continue
        ds = d[sel]
        reach = max(reach, min(abs(key * width), abs((key + 1) * width)))
        n_distinct = torch.unique(x[sel]).numel()
        lim = gelu_fit(torch.tensor(max(abs(key * width), abs((key + 1) * width)))).item() + z * ds.std().item() / n_distinct ** 0.5
        r = abs(ds.mean().item()) / lim
        if r > worst:
            worst, where = r, (key * width, (key + 1) * width, ds.mean().item(), lim, n)
    msg = f"{name}: worst binned-mean ratio {worst:.3g}" + (f" in x in [{where[0]:.2f}, {where[1]:.2f}): mean {where[2]:.3g}, "
                                                          f"limit {where[3]:.3g}, {where[4]} elements" if where else "")
    print(msg + f"; checked bins reach |x| = {reach:.2f}")
    assert worst <= 1.0, msg
    assert reach >= covers, f"{name}: no bin of >= {min_count} elements at |x| >= {covers} (reached {reach:.2f})"
    return worst
