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

import math
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


# --------------------------------------------------------------------------------------------------------------------------------
# the front of a block (casa gate) and the two ends of the trunk (entry, fusion)
# --------------------------------------------------------------------------------------------------------------------------------
EX2_REL = 2.0 ** -22      # ex2.approx.f32: maximum relative error 2 ulp (PTX ISA, ex2)
RCP_REL = 2.0 ** -23      # rcp.approx.f32: maximum error 1 ulp (PTX ISA, rcp)
SIG_FAST = 2.0 ** -11.987  # sigmoid_fast = 0.5 + 0.5 tanh.approx(x / 2): tanh.approx.f32 relative error 2^-10.987 (PTX ISA), halved
SIG_LIP = 0.25            # max |sigmoid'(z)| = 1/4 (z = 0)
SPLIT3 = 2.0 ** -14       # three-term bf16 split of a product a W (glue.cu split_bf16), see `casa_qkv`


def _round_up(n: int, w: int) -> int:
    return (n + w - 1) // w * w


def reflect_pad(x, win: int):
    """Reflect padding of an NHWC map to multiples of `win` (the oracle's index map)."""
    from oracle.hitsir_oracle import reflect_index
    B, H, W, C = x.shape
    return x[:, reflect_index(H, _round_up(H, win))][:, :, reflect_index(W, _round_up(W, win))]


def _split3_conv(a, w, b):
    """fp32 emulation of the casa gate's three-term split contraction (glue.cu:257-261): a_hi W_hi + a_lo W_hi + a_hi W_lo + b_hi + b_lo
    with x_hi = bf16(x), x_lo = bf16(x - x_hi)."""
    def split(t):
        hi = bf(t).float()
        return hi, bf(t.float() - hi).float()
    (ah, al), (wh, wl), (bh, bl) = split(a), split(w), split(b)
    return _conv(ah, wh) + _conv(al, wh) + _conv(ah, wl) + bh + bl


def casa_qkv(x, P, win: int, ar: Arith, mut=()):
    """The casa gate (SpatialChannelAttention, :338-359) as `sca_stats` / `ffn_tail`'s statistics warp + `sca_mlp` +
    `qkv_casa_mma_kernel`: the fp32 block input (B, H, W, 180) -> the gated, reflect-padded bf16 token map (B, Hp, Wp, 180), tap
    `block0.j.qkv`.  Everything reads the fp32 stream and fp32 weights; the arithmetic, element by element:

      global pools over the PADDED map, a pixel counted once per padded position that mirrors it (`reflect_mult`):
          avg: a reduction of Hp Wp terms, / (Hp Wp)          e_avg = Hp Wp 2^-22 mean|xp| + 2^-24 |avg|        max: exact
      Linear 180 -> 18 -> 180 twice, fp32 FMA chains:         e_h = |W_f| e_pool + 181 2^-22 M_f ;  e_s = |W_s| e_h + 19 2^-22 M_s
      channel mean / max per padded pixel (180 terms):        e_cavg = 180 2^-22 mean_c|x| + 2^-24 |cavg|
      3x3 Conv2d(1, 180) over the padded statistic maps (zero outside Hp x Wp, reflected values inside) as ONE bf16 MMA of K = 29
      (glue.cu:257-261): with x_hi = bf16(x), x_lo = bf16(x - x_hi), |x - x_hi| <= 2^-8 |x| and the dropped residual
      |x - x_hi - x_lo| <= 2^-16 |x|, the kernel sums a_hi W_hi + a_lo W_hi + a_hi W_lo, which differs from a W by
      a_hi W_r + a_lo (W_lo + W_r) + a_r W (W_r, a_r the residuals), at most (2^-16 + 2^-16 + 2^-16)(1 + 2^-7) |a||W| < 2^-14 |a||W|; the
      bias loses its residual (2^-16 |b|); the 29 products, at most (1 + 2^-6) |a||W| + |b| in magnitude, are summed in fp32:
          e_conv = |W| * e_stat + 2^-14 |a|*|W| + 2^-16 |b| + 29 2^-22 (1 + 2^-6) M_conv
      LeakyReLU(0.2) as fmaxf(d, 0.2f d) (1-Lipschitz; 0.2f is 0.2 (1 + d), |d| < 2^-26, and the product is rounded: together at most
      2^-23 |0.2 d| on the negative side, which the 29 2^-22 M_conv term of e_conv covers by a factor > 100), then
      o = 0.5 s2 l2 + (0.5 s1 l1 + x) as two fp32 FMAs (the 0.5 is exact):
          e_o = 0.5 (|s1| e_l1 + |l1| e_s1 + e_l1 e_s1 + same for 2) + 2 2^-24 (0.5 |s1 l1| + 0.5 |s2 l2| + |x|)
      and the bf16 store (ulp).  Rounding sites: none besides the split (which SIM evaluates as the kernel does) and the output.
    Mutants: "pool_unpadded" (pools over the unpadded map), "halo_zero" (the gate convs read zeros instead of the reflected
    statistics outside the image), "lrelu_slope" (0.01)."""
    q = "qkv."
    B, H, W, C = x.shape
    slope = 0.01 if "lrelu_slope" in mut else 0.2
    xf = ar.f32(x)
    xp = reflect_pad(xf, win)
    Hp, Wp = xp.shape[1:3]
    inside = torch.zeros(1, Hp, Wp, 1, dtype=torch.bool)
    inside[:, :H, :W] = True
    stats = [xp.mean(-1, keepdim=True), xp.amax(-1, keepdim=True)]
    if "halo_zero" in mut:
        stats = [torch.where(inside, s, torch.zeros_like(s)) for s in stats]
    pools = [(xf if "pool_unpadded" in mut else xp).mean((1, 2)), xp.amax((1, 2))]
    out = xp
    for v, (stat, pool) in enumerate(zip(stats, pools), 1):
        s = _lin(_lin(pool, ar.f32(P[q + f"linear{v}_first.weight"]), ar.f32(P[q + f"linear{v}_first.bias"])),
                 ar.f32(P[q + f"linear{v}_second.weight"]), ar.f32(P[q + f"linear{v}_second.bias"]))
        w, b = P[q + f"linear{v}.weight"], P[q + f"linear{v}.bias"]
        a = _split3_conv(stat, w, b) if ar.bf16_sites else _conv(stat, ar.f32(w), ar.f32(b))
        out = out + F.leaky_relu(a, slope) * s.view(B, 1, 1, C) / 2.0
    out = ar.out(out, True)

    xp64 = reflect_pad(x.double(), win)
    ref = xp64.clone()
    bound = 2 * U32 * xp64.abs()
    stats = [(xp64.mean(-1, keepdim=True), C * UACC * xp64.abs().mean(-1, keepdim=True)),
             (xp64.amax(-1, keepdim=True), torch.zeros(B, Hp, Wp, 1, dtype=torch.float64))]
    stats[0] = (stats[0][0], stats[0][1] + U32 * stats[0][0].abs())
    pools = [(xp64.mean((1, 2)), Hp * Wp * UACC * xp64.abs().mean((1, 2))), (xp64.amax((1, 2)), torch.zeros(B, C, dtype=torch.float64))]
    pools[0] = (pools[0][0], pools[0][1] + U32 * pools[0][0].abs())
    for v, ((stat, e_stat), (pool, e_pool)) in enumerate(zip(stats, pools), 1):
        wf, bf_ = P[q + f"linear{v}_first.weight"].double(), P[q + f"linear{v}_first.bias"].double()
        ws, bs = P[q + f"linear{v}_second.weight"].double(), P[q + f"linear{v}_second.bias"].double()
        h = _lin(pool, wf, bf_)
        e_h = _lin(e_pool, wf.abs()) + _nnz_k(wf) * UACC * _lin(pool.abs(), wf.abs(), bf_.abs())
        s = _lin(h, ws, bs)
        e_s = _lin(e_h, ws.abs()) + _nnz_k(ws) * UACC * _lin(h.abs() + e_h, ws.abs(), bs.abs())
        w, b = P[q + f"linear{v}.weight"].double(), P[q + f"linear{v}.bias"].double()
        a = _conv(stat, w, b)
        m = _conv(stat.abs(), w.abs())
        e_a = _conv(e_stat, w.abs()) + SPLIT3 * m + 2.0 ** -16 * b.abs() + 29 * UACC * (1 + 2.0 ** -6) * (m + b.abs())
        lr = F.leaky_relu(a, 0.2)
        s, e_s = s.view(B, 1, 1, C), e_s.view(B, 1, 1, C)
        ref = ref + 0.5 * s * lr
        bound = bound + 0.5 * (s.abs() * e_a + lr.abs() * e_s + e_a * e_s) + U32 * (s * lr).abs()
    return out, bound + ulp(ref, True)


def entry(x_img, sd, ar: Arith, ms: bool = True, mut=(), img_range=1.0, mean=RGB_MEAN):
    """The image (B, 3, H, W) fp32 -> the shallow features (B, H, W, 180) fp32, tap `shallow` (:1310-1311, :67-100).
    `entry_im2col_kernel` stages bf16((x - mean) * img_range) (fp32 subtract and scale, then one rounding: the operand, exact here),
    zero outside the image (the 9 x 9 footprint of conv9 pads by 4).  Without the multi-size extractor, conv_first is a 3 x 3 conv,
    K = 27 + bias (`conv3`).  With it, one GEMM with the `EPI_MSGATE` epilogue (umma_gemm_tma.cu:259-300) evaluates conv_x (K = 3 + 1)
    and conv3/5/7/9 (K = 3 k^2 + 1; the zero taps of the 9 x 9 footprint add exact zeros), and per output:

        z = x1 x_k (fp32):                 e_z = |x1| e_k + |x_k| e_1 + e_k e_1 + 2^-24 |z|
        sigma = rcp(1 + ex2(-log2e z)):    e_sig = e_z / 4 (sigma is 1/4-Lipschitz)
                                               + sigma (1 - sigma) (2^-22 + 2 2^-24 |z|)   (ex2: PTX max relative error 2 ulp; the rounded
                                                 constant log2e and the rounded product perturb the exponent by 2 2^-24 |log2e z|,
                                                 i.e. 2^(.) by 2 2^-24 |z| relative; a relative error d of ex2 moves sigma by sigma (1 - sigma) d)
                                               + sigma (2^-24 + 2^-23)                    (1 + e rounded, rcp: PTX max error 1 ulp)
        g_k = fma(x_k, sigma, x_k):        e_g = e_k (1 + sigma) + |x_k| e_sig + e_k e_sig + 2^-24 |g_k|
        G = bf16(g_k)                      rounding site 1
        conv_first.conv_last 720 -> 180:  |W_last| * e_G + 721 2^-22 M_last, fp32 store (ulp).
    Mutants: "gate_no_residual" (g_k = x_k sigma), "mean_added" ((x + mean) * img_range)."""
    C = sd["conv_first.conv_last.weight"].shape[0] if ms else sd["conv_first.weight"].shape[0]
    m = torch.tensor(mean, dtype=torch.float32).view(1, -1, 1, 1)
    xf = x_img.float()
    xa, ma = (xf, m) if ar.bf16_operands else (x_img.double(), m.double())
    xs = (((xa + ma) if "mean_added" in mut else (xa - ma)) * img_range).permute(0, 2, 3, 1)
    if not ms:
        return conv3(xs, sd["conv_first.weight"], sd["conv_first.bias"], ar)
    p = "conv_first."
    op = ar.op(xs)
    x1 = _conv(op, ar.op(sd[p + "conv_x.weight"]), ar.f32(sd[p + "conv_x.bias"]), 0)
    gs = []
    for k in (3, 5, 7, 9):
        xk = _conv(op, ar.op(sd[p + f"conv{k}.weight"]), ar.f32(sd[p + f"conv{k}.bias"]), k // 2)
        g = xk * torch.sigmoid(x1 * xk)
        gs.append(ar.site(g if "gate_no_residual" in mut else g + xk))
    wl, bl = sd[p + "conv_last.weight"], sd[p + "conv_last.bias"]
    out = _lin(torch.cat(gs, -1), ar.op(wl.reshape(C, -1)), ar.f32(bl))

    op64 = bf(((xf - m) * img_range).permute(0, 2, 3, 1))
    wx, bx = bf(sd[p + "conv_x.weight"]), sd[p + "conv_x.bias"].double()
    x1 = _conv(op64, wx, bx, 0)
    e1 = _nnz_k(wx) * UACC * _conv(op64.abs(), wx.abs(), bx.abs(), 0)
    g64, eg = [], []
    for k in (3, 5, 7, 9):
        wk, bk = bf(sd[p + f"conv{k}.weight"]), sd[p + f"conv{k}.bias"].double()
        xk = _conv(op64, wk, bk, k // 2)
        ek = _nnz_k(wk) * UACC * _conv(op64.abs(), wk.abs(), bk.abs(), k // 2)
        z = x1 * xk
        ez = x1.abs() * ek + xk.abs() * e1 + ek * e1 + U32 * z.abs()
        sig = torch.sigmoid(z)
        es = SIG_LIP * ez + sig * (1 - sig) * (EX2_REL + 2 * U32 * z.abs()) + sig * (U32 + RCP_REL)
        g = xk * sig + xk
        g64.append(g)
        eg.append(_site(ek * (1 + sig) + xk.abs() * es + ek * es + U32 * g.abs(), g))
    G, eG = torch.cat(g64, -1), torch.cat(eg, -1)
    wl64 = bf(wl.reshape(C, -1))
    ref = _lin(G, wl64, bl.double())
    bound = _lin(eG, wl64.abs()) + _nnz_k(wl64) * UACC * _lin(G.abs() + eG, wl64.abs(), bl.double().abs())
    return out, bound + ulp(ref, False)


def _conv2to1(pa, pm, w, b, mut=()):
    """Conv2d(2, 1, 3, padding=1) on a (B, R, S) plane pair (mean plane first, as torch.cat((mean, max)) stacks them)."""
    if "planes_swapped" in mut:
        pa, pm = pm, pa
    return F.conv2d(torch.stack((pa, pm), 1), w, b, 1, 1)[:, 0]


def _ua_stats(X):
    """channel mean / max per pixel (B, H, W), mean / max over H per (channel, x) (B, C, W), over W per (channel, y) (B, C, H)."""
    return (X.mean(-1), X.amax(-1), X.mean(1).transpose(1, 2), X.amax(1).transpose(1, 2), X.mean(2).transpose(1, 2),
            X.amax(2).transpose(1, 2))


def union_attention(X, sd, p: str, ar: Arith, mut=()):
    """UnionAttention (:113-133) as `ua_rows` + `ua_cols` + `ua_small_convs` + `ua_build` + `conv_ua`, evaluated under `ar`."""
    ca, cm, ha, hm, wa, wm = _ua_stats(X)
    w3 = sd[p + "conv3.weight"]
    if "ch_h_not_transposed" in mut:
        w3 = w3.transpose(-1, -2)
    c_att = _conv2to1(ca, cm, ar.f32(sd[p + "conv1.weight"]), ar.f32(sd[p + "conv1.bias"]), mut)
    h_att = _conv2to1(ha, hm, ar.f32(sd[p + "conv2.weight"]), ar.f32(sd[p + "conv2.bias"]), mut)
    w_att = _conv2to1(wa, wm, ar.f32(w3), ar.f32(sd[p + "conv3.bias"]), mut)
    s = ar.site(c_att[..., None] + w_att.transpose(1, 2)[:, :, None, :] + h_att.transpose(1, 2)[:, None, :, :])
    return _conv(s, ar.op(sd[p + "conv_last.weight"]), ar.f32(sd[p + "conv_last.bias"]))


def union_attention_bound(X, eX, sd, p: str):
    """(exact UnionAttention of X in float64 with the kernel's operands, bound of the kernel's error given |X~ - X| <= eX):
      statistics: a mean of n fp32 terms (n = C, W or H): mean(eX) + n 2^-22 mean|X| + 2^-24 |mean|; a max: max(eX)
      each 2 -> 1 3x3 conv (fp32, K = 18 + 1, zero padding):  |w| * e_stat + 19 2^-22 M
      s = c_att + w_att + h_att (two fp32 adds), stored bf16 (rounding site 1); conv_ua 3x3 180 -> 180 on the bf16 s (K = 1620 + 1)."""
    B, H, W, C = X.shape
    A = X.abs()
    st = _ua_stats(X)
    es = (eX.mean(-1) + C * UACC * A.mean(-1) + U32 * st[0].abs(), eX.amax(-1),
          eX.mean(1).transpose(1, 2) + H * UACC * A.mean(1).transpose(1, 2) + U32 * st[2].abs(), eX.amax(1).transpose(1, 2),
          eX.mean(2).transpose(1, 2) + W * UACC * A.mean(2).transpose(1, 2) + U32 * st[4].abs(), eX.amax(2).transpose(1, 2))
    att, e_att = [], []
    for i, k in enumerate(("conv1", "conv2", "conv3")):
        w, b = sd[p + k + ".weight"].double(), sd[p + k + ".bias"].double()
        att.append(_conv2to1(st[2 * i], st[2 * i + 1], w, b))
        e_att.append(_conv2to1(es[2 * i], es[2 * i + 1], w.abs(), None) +
                     19 * UACC * _conv2to1(st[2 * i].abs(), st[2 * i + 1].abs(), w.abs(), b.abs()))

    def build(c, h, w_):
        return c[..., None] + w_.transpose(1, 2)[:, :, None, :] + h.transpose(1, 2)[:, None, :, :]
    s = build(*att)
    e_s = _site(build(*e_att) + 2 * U32 * build(*[a.abs() for a in att]), s)
    w, b = bf(sd[p + "conv_last.weight"]), sd[p + "conv_last.bias"].double()
    a = _conv(s, w, b)
    return a, _conv(e_s, w.abs()) + _nnz_k(w) * UACC * _conv(s.abs() + e_s, w.abs(), b.abs())


def fusion(cab, shallow, sd, ar: Arith, mut=()):
    """Fusion.forward (:145-162) with the positional binding of :1330: first = conv_after_body, second = shallow (both fp32 maps,
    taps `conv_after_body` and `shallow`) -> the fp32 map `fusion_combine` writes (tap `fused`) before its bf16 store.  Three
    UnionAttentions (`union_attention_bound`; the second on first + second, one fp32 add), then `fusion_combine_kernel` with
    sigmoid_fast (absolute error <= 2^-11.987 plus the fp32 FMA, 1/4-Lipschitz):
        t = sig(a2):                  e_t = e_a2 / 4 + 2^-11.987 + 2^-24
        u1 = a1 t, u3 = a3 (1 - t):   e_u = |a| e_t' + |t'| e_a + e_a e_t' + 2^-24 |u|   (1 - t rounded: e_t' = e_t + 2^-24)
        out = f sig(u1) + s sig(u3):  |f| e_sig1 + |s| e_sig3 + 2 2^-24 (|f sig1| + |s sig3|)      (fp32 multiply + FMA)
    Mutants: "swap" (first and second exchanged), "sig_outside" (sig(a1) t), "ch_h_not_transposed", "planes_swapped"."""
    p = "fusion.union_attention"
    first, second = (shallow, cab) if "swap" in mut else (cab, shallow)
    f, s = ar.f32(first), ar.f32(second)
    a1 = union_attention(f, sd, p + "1.", ar, mut)
    t = torch.sigmoid(union_attention(f + s, sd, p + "2.", ar, mut))
    a3 = union_attention(s, sd, p + "3.", ar, mut)
    g1 = torch.sigmoid(a1) * t if "sig_outside" in mut else torch.sigmoid(a1 * t)
    out = f * g1 + s * torch.sigmoid(a3 * (1 - t))

    f, s = cab.double(), shallow.double()
    a1, e1 = union_attention_bound(f, torch.zeros_like(f), sd, p + "1.")
    a2, e2 = union_attention_bound(f + s, U32 * (f + s).abs(), sd, p + "2.")
    a3, e3 = union_attention_bound(s, torch.zeros_like(s), sd, p + "3.")
    t = torch.sigmoid(a2)
    e_t = SIG_LIP * e2 + SIG_FAST + U32
    u1, u3 = a1 * t, a3 * (1 - t)
    e_u1 = a1.abs() * e_t + t * e1 + e1 * e_t + U32 * u1.abs()
    e_u3 = a3.abs() * (e_t + U32) + (1 - t) * e3 + e3 * (e_t + U32) + U32 * u3.abs()
    g1, g3 = torch.sigmoid(u1), torch.sigmoid(u3)
    ref = f * g1 + s * g3
    bound = f.abs() * (SIG_LIP * e_u1 + SIG_FAST + U32) + s.abs() * (SIG_LIP * e_u3 + SIG_FAST + U32) + 2 * U32 * ((f * g1).abs() + (s * g3).abs())
    return out, bound + ulp(ref, False)


# --------------------------------------------------------------------------------------------------------------------------------
# window self-correlation (S-SC + C-SC without proj)
# --------------------------------------------------------------------------------------------------------------------------------
HEADS, HD = 6, 15


def _pool_geom(P, win: int):
    """(pooled grid side, pooling ratio r) of a window, read off spatial_linear = Linear(r^2, 1): base = min(w, base_win_size)."""
    r = math.isqrt(P["spatial_linear.weight"].numel())
    return win // r, r


def _scc_operands(P, win: int, ar: Arith, mut=()):
    """The weight operands of both SCC kernels: the k-gen image (`scc_w_image_kernel`) holds bf16(0.5 w1), bf16(0.5 w2) and
    bf16(0.5 (b1 + b2)) (fp32 sum, on the ones column of each head's q slice); the pool weights are a bf16 operand image when r > 1
    (`scc_pool_image_kernel`) and an fp32 scalar in `scc_dense`; spatial_linear.bias is an fp32 scalar.  Returns (W1x [15, 16] =
    [W1 | bk], W2 [15, 15], pool matrix [L, Lb], bsl)."""
    w1, w2 = P["k_generate1.weight"], P["k_generate2.weight"]
    b1, b2 = P["k_generate1.bias"], P["k_generate2.bias"]
    if "kgen_swapped" in mut:
        w1, w2, b1, b2 = w2, w1, b2, b1
    bk = 0.5 * (b1.float() + b2.float())
    if "no_ones" in mut:
        bk = torch.zeros_like(bk)
    W1x = torch.cat([ar.op(0.5 * w1.float()), ar.op(bk)[:, None]], 1)
    W2 = ar.op(0.5 * w2.float())
    base, r = _pool_geom(P, win)
    wsl = P["spatial_linear.weight"].reshape(-1)
    wsl = ar.op(wsl) if r > 1 else ar.f32(wsl)
    ly, lx = torch.div(torch.arange(win * win), win, rounding_mode="floor"), torch.arange(win * win) % win
    pool = torch.zeros(win * win, base * base, dtype=ar.dtype)
    pool[torch.arange(win * win), (ly // r) * base + lx // r] = wsl[(ly % r) * r + lx % r].to(ar.dtype)
    return W1x, W2, pool, ar.f32(P["spatial_linear.bias"].reshape(()))


def _win_qv(tok, win: int, dtype):
    """Padded token map (B, Hp, Wp, 180) -> per-window q with the ones column (n, L, 6, 16) and v (n, L, 6, 15)."""
    from oracle.hitsir_oracle import to_windows
    tw = to_windows(tok.to(dtype), (win, win))
    n, L, _ = tw.shape
    q = tw[..., :HEADS * HD].reshape(n, L, HEADS, HD)
    return torch.cat([q, torch.ones(n, L, HEADS, 1, dtype=dtype)], -1), tw[..., HEADS * HD:].reshape(n, L, HEADS, HD)


def _kgen(xq, xv, W1x, W2):
    """k-gen applied along the last axis: xq has 16 entries (ones column), xv 15."""
    return xq @ W1x.t() + xv @ W2.t()


def _scc_out(out_s, out_c, tok, win, hw):
    from oracle.hitsir_oracle import from_windows
    B, Hp, Wp, _ = tok.shape
    n, L = out_s.shape[:2]
    out = torch.cat([out_s.reshape(n, L, -1), out_c.reshape(n, L, -1)], -1)
    return from_windows(out, (win, win), B, Hp, Wp)[:, :hw[0], :hw[1]]


def _scc_ref(tok, bias, P, win, ar: Arith, mut=()):
    """SCC.forward without proj (oracle/hitsir_oracle.py:185-213) evaluated directly under `ar` with the kernel's operands."""
    W1x, W2, pool, bsl = _scc_operands(P, win, ar, mut)
    qh, v = _win_qv(tok, win, ar.dtype)
    q = qh[..., :HD]
    L = win * win
    k = _kgen(qh, v, W1x, W2)
    kp = torch.einsum("lm,nlhj->nmhj", pool, k) + bsl
    vp = torch.einsum("lm,nlhj->nmhj", pool, v) + bsl
    bias = ar.op(bias)
    corr = torch.einsum("nlhj,nmhj->nhlm", q, kp) / HD + bias
    out_s = torch.einsum("nhlm,nmhd->nlhd", corr, vp)
    qm, km, vm = q.reshape(*q.shape[:2], -1), k.reshape(*k.shape[:2], -1), v.reshape(*v.shape[:2], -1)
    out_c = torch.einsum("nlc,nle,nme->nmc", qm, km, vm) / L
    return out_s, out_c


def _scc_umma_sim(tok, bias, P, win, mut=()):
    """scc_umma in fp32 with its bf16 sites: G = Q^T T, TPT (raw pooled tokens), VPT = pooled v + bsl, corr = G Wk^T / L, KP =
    Wk TPT + bsl, Mblk = KP_h^T VP_h / 15; out_s = Q Mblk + sum_m bias VP, out_c = V corr^T."""
    ar = SIM
    W1x, W2, pool, bsl = _scc_operands(P, win, ar, mut)
    qh, v = _win_qv(tok, win, torch.float32)
    q = qh[..., :HD]
    L = win * win
    Gq = ar.site(torch.einsum("nlhi,nlgj->nhigj", q, qh))
    Gv = ar.site(torch.einsum("nlhi,nlgj->nhigj", q, v))
    inv_l = 1.0 / (pool.shape[1] if "inv_lb" in mut else L)
    corr = ar.site(_kgen(Gq, Gv, W1x, W2) * torch.tensor(inv_l, dtype=torch.float32))
    out_c = torch.einsum("nlgj,nhigj->nlhi", v, corr)
    tq = ar.site(torch.einsum("lm,nlhi->nmhi", pool, qh))
    tv_raw = torch.einsum("lm,nlhi->nmhi", pool, v)
    tv = ar.site(tv_raw)
    vpt = ar.site(tv_raw if "no_bsl_vpt" in mut else tv_raw + bsl)
    kp = ar.site(_kgen(tq, tv, W1x, W2) + (0.0 if "no_bsl_kp" in mut else bsl))
    scale = torch.tensor(1.0 / (16 if "scale16" in mut else 15), dtype=torch.float32)
    mblk = ar.site(torch.einsum("nmhj,nmhd->nhjd", kp, vpt) * scale)
    b = ar.op(bias)
    if "bias_xy" in mut:
        b = b.reshape(HEADS, win, win, -1).transpose(1, 2).reshape(b.shape)
    out_s = torch.einsum("nlhj,nhjd->nlhd", q, mblk) + torch.einsum("hlm,nmhd->nlhd", b, vpt)
    return out_s, out_c


def _scc_dense_sim(tok, bias, P, win, mut=()):
    """scc_dense in fp32 with its bf16 sites: K = T Wk^T (bf16 K tile); C-SC P_c = bf16(mask(V K^T) / L), out_c = P_c Q;
    S-SC val = (a S_h + b sum_i q_i) / 15 + bias_h, P_h = bf16(val), out_s = a P_h V_h + b rowsum(val)."""
    ar = SIM
    W1x, W2, pool, bsl = _scc_operands(P, win, ar, mut)
    a = pool.sum(0)[0]
    qh, v = _win_qv(tok, win, torch.float32)
    q = qh[..., :HD]
    L = win * win
    K = ar.site(_kgen(qh, v, W1x, W2))
    n = q.shape[0]
    st = torch.einsum("nle,nme->nlm", v.reshape(n, L, -1), K.reshape(n, L, -1))
    pc = ar.site(st / (pool.shape[1] if "inv_lb" in mut else L))
    out_c = torch.einsum("nlm,nmc->nlc", pc, q.reshape(n, L, -1)).reshape(n, L, HEADS, HD)
    inv15 = torch.tensor(1.0 / (16 if "scale16" in mut else 15), dtype=torch.float32)
    S = torch.einsum("nlhj,nmhj->nhlm", q, K)
    qsum = q.sum(-1).permute(0, 2, 1)[..., None]
    b = ar.op(bias)
    if "bias_transposed" in mut:
        b = b.transpose(1, 2)
    val = (a * inv15) * S + (0.0 if "no_bsl_kp" in mut else bsl * qsum * inv15) + b
    D = torch.einsum("nhlm,nmhd->nlhd", ar.site(val), v)
    rs = val.sum(-1).permute(0, 2, 1)[..., None]
    out_s = a * D + (0.0 if "no_bsl_vpt" in mut else bsl * rs)
    return out_s, out_c


def scc(tok, bias, P, win: int, ar: Arith, hw, mut=()):
    """The window self-correlation without proj: the padded bf16 token map (B, Hp, Wp, 180; tap `block0.j.qkv`, exact) and the
    device's fp32 pooled bias table (6, L, Lb; read as a bf16 operand) -> the cropped bf16 output (B, H, W, 180; tap `block0.j.scc`).
    REF/PIN evaluate SCC.forward directly; SIM evaluates the kernel's own re-association (`scc_umma` for r > 1, `scc_dense` for r = 1).
    The bound is the kernel's, per output element of a window (n = window, l = token, h = head; |.| magnitude passes on the exact REF
    operands, e_X the carried error of an intermediate X, `_site` its bf16 rounding):

    scc_umma (header of scc_umma.cu), sites G, TPT, VPT, corr, KP, Mblk and the output:
        G = Q^T T (L terms):                e_G = site(L 2^-22 |Q|^T |T|)
        corr = bf16(G Wk^T * fl(1/L)):      e_corr = site((|Wk| e_G + 32 2^-22 |Wk| (|G| + e_G)) / L + 2 2^-24 |corr|)
                                            (1/L rounded to fp32 and the product: 2 2^-24; |G| is carried, not |corr|)
        out_c = V corr^T (96 terms):        |V| e_corr + 96 2^-22 |V| (|corr| + e_corr)
        TPT = Pool^T T (r^2 terms):         e_TPT = site(r^2 2^-22 |Pool|^T |T|)
        VPT = bf16(pooled v + bsl):         e_VPT = site(r^2 2^-22 |Pool|^T |V| + 2^-24 |VPT|)
        KP = bf16(Wk TPT + bsl):            e_KP = site(|Wk| e_TPT + 32 2^-22 |Wk| (|TPT| + e_TPT) + 2^-24 |KP|)
        Mblk = bf16(KP_h^T VP_h * fl(1/15)): e_M = site((e_KP|VPT| + |KP| e_VPT + e_KP e_VPT + Lb 2^-22 (|KP|+e)(|VPT|+e)) / 15
                                                          + 2 2^-24 |M|)
        out_s = Q Mblk + bias VPT (16 + 64 terms):  |Q| e_M + |bias| e_VPT + 80 2^-22 (|Q| (|M|+e_M) + |bias| (|VPT|+e_VPT))
    scc_dense (header of scc_dense.cu), sites K, P_c, P_h and the output; a = spatial_linear.weight, b = its bias (fp32):
        K = bf16(T Wk^T) (31 terms):        e_K = site(32 2^-22 |Wk| |T|)
        P_c = bf16(V K^T / L) (96 terms, L a power of two):  e_Pc = site((|V| e_K^T + 96 2^-22 |V| (|K| + e_K)^T) / L)
        out_c = P_c Q (L terms):            e_Pc |Q| + L 2^-22 (|P_c| + e_Pc) |Q|
        S_h = Q_h K_h^T (16 terms):         e_S = |Q_h| e_K^T + 16 2^-22 |Q_h| (|K_h| + e_K)^T
        val = fma(fl(a fl(1/15)), S, fl(fl(b qsum) fl(1/15))) + bias, qsum a 15-term fp32 sum: at most 18 roundings along any path,
                                            e_val = |a| e_S / 15 + 18 2^-24 (|a S| / 15 + |b| sum|q| / 15 + |bias|)
        P_h = bf16(val):                    e_P = site(e_val)
        out_s = fma(a, P_h V_h, b rowsum(val)) with rowsum over the UNROUNDED val (L terms):
                                            |a| (e_P |V| + L 2^-22 (|P|+e_P) |V|) + |b| (sum e_val + L 2^-22 sum(|val|+e_val))
                                            + 2 2^-24 (|a D| + |b rowsum|)
    and one bf16 ulp of the stored output.  Mutants of SIM: "no_bsl_vpt", "no_bsl_kp", "scale16", "inv_lb", "kgen_swapped",
    "no_ones", "bias_transposed" (scc_dense: the L x L table read (m, l)), "bias_xy" (scc_umma: the L x Lb table's token rows read
    with x and y exchanged -- an (m, l) read of a non-square table is not a plausible kernel bug)."""
    base, r = _pool_geom(P, win)
    if ar is SIM:
        out_s, out_c = (_scc_dense_sim if r == 1 else _scc_umma_sim)(tok, bias, P, win, mut)
    else:
        out_s, out_c = _scc_ref(tok, bias, P, win, ar, mut)
    out = ar.out(_scc_out(out_s, out_c, tok, win, hw), True)

    W1x, W2, pool, bsl = _scc_operands(P, win, REF)
    A1, A2, Ap, bsl_a = W1x.abs(), W2.abs(), pool.abs(), abs(bsl.item())
    qh, v = _win_qv(tok, win, torch.float64)
    q = qh[..., :HD]
    aq, aqh, av = q.abs(), qh.abs(), v.abs()
    L, Lb = win * win, base * base
    ref_s, ref_c = _scc_ref(tok, bias, P, win, REF)
    bias = bf(bias)
    n = q.shape[0]
    if r > 1:
        G = [torch.einsum("nlhi,nlgj->nhigj", q, x) for x in (qh, v)]
        eG = [_site(L * UACC * torch.einsum("nlhi,nlgj->nhigj", aq, x), g) for x, g in zip((aqh, av), G)]
        corr = _kgen(G[0], G[1], W1x, W2) / L
        e_corr = _site((_kgen(eG[0], eG[1], A1, A2) + 32 * UACC * _kgen(G[0].abs() + eG[0], G[1].abs() + eG[1], A1, A2)) / L
                       + 2 * U32 * corr.abs(), corr)
        e_c = torch.einsum("nlgj,nhigj->nlhi", av, e_corr) + 96 * UACC * torch.einsum("nlgj,nhigj->nlhi", av, corr.abs() + e_corr)
        tq, tv = (torch.einsum("lm,nlhi->nmhi", pool, x) for x in (qh, v))
        e_tq, e_tv = (_site(r * r * UACC * torch.einsum("lm,nlhi->nmhi", Ap, x), t) for x, t in ((aqh, tq), (av, tv)))
        vpt = tv + bsl
        e_vpt = _site(r * r * UACC * torch.einsum("lm,nlhi->nmhi", Ap, av) + U32 * vpt.abs(), vpt)
        kp = _kgen(tq, tv, W1x, W2) + bsl
        e_kp = _site(_kgen(e_tq, e_tv, A1, A2) + 32 * UACC * (_kgen(tq.abs() + e_tq, tv.abs() + e_tv, A1, A2) + bsl_a)
                     + U32 * kp.abs(), kp)
        M = torch.einsum("nmhj,nmhd->nhjd", kp, vpt) / HD
        e_M = _site((torch.einsum("nmhj,nmhd->nhjd", e_kp, vpt.abs()) + torch.einsum("nmhj,nmhd->nhjd", kp.abs() + e_kp, e_vpt)
                     + Lb * UACC * torch.einsum("nmhj,nmhd->nhjd", kp.abs() + e_kp, vpt.abs() + e_vpt)) / HD + 2 * U32 * M.abs(), M)
        ab = bias.abs()
        e_s = (torch.einsum("nlhj,nhjd->nlhd", aq, e_M) + torch.einsum("hlm,nmhd->nlhd", ab, e_vpt)
               + 80 * UACC * (torch.einsum("nlhj,nhjd->nlhd", aq, M.abs() + e_M) + torch.einsum("hlm,nmhd->nlhd", ab, vpt.abs() + e_vpt)))
    else:
        a, b = pool.sum(0)[0].item(), bsl.item()
        K = _kgen(qh, v, W1x, W2)
        e_K = _site(32 * UACC * _kgen(aqh, av, A1, A2), K)
        vm, avm, Km, e_Km = (x.reshape(n, L, -1) for x in (v, av, K, e_K))
        st = torch.einsum("nle,nme->nlm", vm, Km)
        e_pc = _site((torch.einsum("nle,nme->nlm", avm, e_Km) + 96 * UACC * torch.einsum("nle,nme->nlm", avm, Km.abs() + e_Km)) / L,
                     st / L)
        aqm = aq.reshape(n, L, -1)
        e_c = (torch.einsum("nlm,nmc->nlc", e_pc, aqm) + L * UACC * torch.einsum("nlm,nmc->nlc", (st / L).abs() + e_pc, aqm))
        e_c = e_c.reshape(n, L, HEADS, HD)
        S = torch.einsum("nlhj,nmhj->nhlm", q, K)
        e_S = torch.einsum("nlhj,nmhj->nhlm", aq, e_K) + 16 * UACC * torch.einsum("nlhj,nmhj->nhlm", aq, K.abs() + e_K)
        aqsum = aq.sum(-1).permute(0, 2, 1)[..., None]
        val = a / HD * S + b * q.sum(-1).permute(0, 2, 1)[..., None] / HD + bias
        e_val = abs(a) * e_S / HD + 18 * U32 * (abs(a) * S.abs() / HD + abs(b) * aqsum / HD + bias.abs())
        e_P = _site(e_val, val)
        D = torch.einsum("nhlm,nmhd->nlhd", val, v)
        e_D = torch.einsum("nhlm,nmhd->nlhd", e_P, av) + L * UACC * torch.einsum("nhlm,nmhd->nlhd", val.abs() + e_P, av)
        rs = val.sum(-1).permute(0, 2, 1)[..., None]
        e_rs = (e_val.sum(-1) + L * UACC * (val.abs() + e_val).sum(-1)).permute(0, 2, 1)[..., None]
        e_s = abs(a) * e_D + abs(b) * e_rs + 2 * U32 * ((a * D).abs() + (b * rs).abs())
    ref = _scc_out(ref_s, ref_c, tok, win, hw)
    return out, _scc_out(e_s, e_c, tok, win, hw) + ulp(ref, True)
