"""Round-2 golden vectors from the UNMODIFIED reference module (run where /root/reference exists):

    python tests/golden/make_golden_r2.py [big] [small] [scc]

* big   -- BASELINE-size inputs (BASELINE.json configs[2] tile 576x576 x2 'pixelshuffle', configs[3] image 512x512 x4
           'nearest+conv'), init and stress weights.  The full outputs are 16-50 MB, so the fixture keeps a prime-strided sample of
           the flattened output, four full-resolution crops and the output moments.
* small -- in_chans = 1 (single-channel images: mean = 0, hit_sir_pro.py:1130-1131), full output.
* scc   -- the pieces of SCC.forward (hit_sir_pro.py:542-599) one by one for all six window sizes: the pooled relative-position bias
           (6, L, Lb) of :477-503, the spatial self-correlation (:458-513) and the channel self-correlation (:515-540) in image order.
           The bias is an intermediate of `spatial_self_correlation`; it is read out of the unmodified method with a linear probe
           (q = 0, pooled v = one-hot, pooling replaced by the identity on the probe instance), so every value is the reference's
           own fp32 number.  S-SC / C-SC are the return values of the reference's methods (recorded by wrapping the bound methods),
           passed through the reference's `window_reverse` and cropped like :696.
"""
import contextlib
import io
import os
import sys
import warnings

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "oracle", "ref_shim"))
sys.path.insert(0, "/root/reference")
sys.path.insert(0, ROOT)
warnings.filterwarnings("ignore")

from oracle.weights import fill_state_dict, synthetic_image  # noqa: E402

with contextlib.redirect_stdout(io.StringIO()):
    import models.hit_sir_pro as ref_mod  # noqa: E402
    from models.hit_sir_pro import HiT_SIR  # noqa: E402

PRO = dict(embed_dim=180, base_win_size=[8, 8], depths=[6] * 6, num_heads=[6] * 6, mlp_ratio=2,
           hier_win_ratios=[0.5, 1, 2, 4, 6, 8, 10, 12])

BIG = [
    # name, flags, upsampler, upscale, mode, wseed, (B,H,W), xseed, stride, crop
    ("big_cfg3_tile576_x2ps_init", (True, True, True), "pixelshuffle", 2, "init", 11, (1, 576, 576), 21, 97, 96),
    ("big_cfg3_tile576_x2ps_stress", (True, True, True), "pixelshuffle", 2, "stress", 12, (1, 576, 576), 22, 97, 96),
    ("big_cfg4_512_x4_init", (True, True, True), "nearest+conv", 4, "init", 13, (1, 512, 512), 23, 257, 128),
    ("big_cfg4_512_x4_stress", (True, True, True), "nearest+conv", 4, "stress", 14, (1, 512, 512), 24, 257, 128),
]


def build(flags, up, scale, mode, wseed, in_chans=3, **extra):
    with contextlib.redirect_stdout(io.StringIO()):
        m = HiT_SIR(*flags, upsampler=up, upscale=scale, in_chans=in_chans, **PRO, **extra).eval()
    sd = fill_state_dict(m.state_dict(), wseed, mode)
    if "absolute_pos_embed" in sd:             # make the embedding matter (its init-like fill is ~1e-3)
        g = torch.Generator().manual_seed(wseed)
        sd["absolute_pos_embed"] = torch.randn(sd["absolute_pos_embed"].shape, generator=g) * 0.5
    m.load_state_dict(sd, strict=True)
    return m, sd


# constructor variants of section 8f-4: name, flags, upsampler, upscale, extra kwargs, (B,H,W), wseed, xseed
VARIANTS = [
    ("var_3conv_x2_direct_40x44", (False, True, True), "pixelshuffledirect", 2, dict(resi_connection="3conv"), (1, 40, 44), 31, 41),
    ("var_ape_x2_direct_40x40", (False, True, True), "pixelshuffledirect", 2, dict(ape=True, img_size=40), (2, 40, 40), 32, 42),
    ("var_noupsampler_40x44", (True, True, True), None, 4, dict(), (1, 40, 44), 33, 43),       # denoise mode: output is x-sized
]


def make_variants():
    for name, flags, up, scale, extra, shape, wseed, xseed in VARIANTS:
        m, sd = build(flags, up, scale, "stress", wseed, **extra)
        x = synthetic_image(*shape, seed=xseed)
        with torch.no_grad():
            y = m(x)
            with torch.autocast("cpu", dtype=torch.bfloat16):
                yb = m(x).float()
        sc = max(1.0, y.abs().max().item())
        import math
        yard = [(y - yb).abs().max().item() / sc, 10.0 * math.log10(1.0 / (((y - yb) / sc).double() ** 2).mean().item())]
        meta = dict(flags=list(flags), upsampler=up, upscale=scale, mode="stress", wseed=wseed, shape=list(shape), xseed=xseed, extra=extra)
        np.savez_compressed(os.path.join(HERE, name + ".npz"), y=y.numpy(), meta=np.array(repr(meta)), yardstick=np.array(yard),
                            keys=np.array("\n".join(f"{k} {tuple(v.shape)}" for k, v in m.state_dict().items())))
        print(f"{name}: y {tuple(y.shape)} mean {y.mean():.6f} std {y.std():.6f} keys {len(sd)} autocast-bf16 {yard}", flush=True)


def crop_origins(hh, ww, c):
    """Four crops: top-left, bottom-right, centre, and one across the middle of the right edge."""
    return [(0, 0), (hh - c, ww - c), ((hh - c) // 2, (ww - c) // 2), ((hh - c) // 2 + 7, ww - c)]


def make_big():
    for name, flags, up, scale, mode, wseed, shape, xseed, stride, crop in BIG:
        m, _ = build(flags, up, scale, mode, wseed)
        x = synthetic_image(*shape, seed=xseed)
        with torch.no_grad():
            y = m(x)
        hh, ww = y.shape[2], y.shape[3]
        arrays = {"sample": y.reshape(-1)[::stride].numpy().copy(), "stride": np.int64(stride),
                  "mean": np.float64(y.double().mean().item()), "std": np.float64(y.double().std().item()),
                  "absmax": np.float64(y.abs().max().item()), "crop": np.int64(crop),
                  "origins": np.array(crop_origins(hh, ww, crop), dtype=np.int64)}
        for i, (y0, x0) in enumerate(crop_origins(hh, ww, crop)):
            arrays[f"crop{i}"] = y[0, :, y0:y0 + crop, x0:x0 + crop].numpy().copy()
        meta = dict(flags=list(flags), upsampler=up, upscale=scale, mode=mode, wseed=wseed, shape=list(shape), xseed=xseed, in_chans=3)
        arrays["meta"] = np.array(repr(meta))
        path = os.path.join(HERE, name + ".npz")
        np.savez_compressed(path, **arrays)
        print(f"{name}: y {tuple(y.shape)} mean {y.mean():.6f} std {y.std():.6f} -> {os.path.getsize(path) / 1e3:.0f} kB", flush=True)


def make_small():
    name, flags, up, scale, mode, wseed, shape, xseed = "gray_x4_direct_40x44", (False, True, True), "pixelshuffledirect", 4, "stress", 15, (2, 40, 44), 25
    m, sd = build(flags, up, scale, mode, wseed, in_chans=1)
    x = synthetic_image(*shape, seed=xseed, chans=1)
    with torch.no_grad():
        y = m(x)
    meta = dict(flags=list(flags), upsampler=up, upscale=scale, mode=mode, wseed=wseed, shape=list(shape), xseed=xseed, in_chans=1)
    np.savez_compressed(os.path.join(HERE, name + ".npz"), y=y.numpy(), meta=np.array(repr(meta)),
                        keys=np.array("\n".join(f"{k} {tuple(v.shape)}" for k, v in m.state_dict().items())))
    print(f"{name}: y {tuple(y.shape)} mean {y.mean():.6f} std {y.std():.6f} keys {len(sd)}", flush=True)


def probe_bias(scc):
    """The (heads, L, Lb) tensor `relative_position_bias` of hit_sir_pro.py:477-503, read through the unmodified method."""
    heads = scc.num_heads
    wh, ww = scc.window_size
    L = wh * ww
    Lb = scc.base_win_size[0] * scc.base_win_size[1]
    hd = scc.dim // (2 * heads)
    nb = -(-Lb // hd)
    q = torch.zeros(nb, heads, L, hd)
    v = torch.zeros(nb, heads, Lb, hd)
    for b in range(nb):
        for j in range(hd):
            if b * hd + j < Lb:
                v[b, :, b * hd + j, j] = 1.0
    saved = scc.spatial_linear_projection
    scc.spatial_linear_projection = lambda t: t          # the probe feeds pooled tensors directly
    try:
        with torch.no_grad():
            out = scc.spatial_self_correlation(q, v.clone(), v)      # (nb, L, heads*hd): out[b,l,h*hd+j] = bias[h,l,b*hd+j]
    finally:
        scc.spatial_linear_projection = saved
    out = out.view(nb, L, heads, hd).permute(2, 1, 0, 3).reshape(heads, L, nb * hd)[:, :, :Lb]
    return out.contiguous()


def make_scc():
    name, flags, mode, wseed, shape, xseed = "scc_parts_56x72", (True, True, True), "stress", 21, (1, 56, 72), 4
    m, _ = build(flags, "nearest+conv", 4, mode, wseed)
    x = synthetic_image(*shape, seed=xseed)
    H, W = shape[1], shape[2]
    rec = {}
    blocks = m.layers[0].residual_group.blocks
    restore = []
    for j, blk in enumerate(blocks):
        scc = blk.correlation
        for kind, meth in (("ssc", "spatial_self_correlation"), ("csc", "channel_self_correlation")):
            orig = getattr(scc, meth)

            def wrapped(q, k, v, orig=orig, key=f"{kind}{j}"):
                out = orig(q, k, v)
                rec[key] = out.detach()
                return out
            setattr(scc, meth, wrapped)
            restore.append((scc, meth))
    with torch.no_grad():
        m(x)
    for scc, meth in restore:
        delattr(scc, meth)                                # back to the class's unmodified bound method
    arrays = {}
    S_STRIDE, B_STRIDE = 26, 34                           # keeps the fixture under 1 MB
    for j, blk in enumerate(blocks):
        scc = blk.correlation
        wh, ww = scc.window_size
        Hp, Wp = -(-H // wh) * wh, -(-W // ww) * ww
        for kind in ("ssc", "csc"):
            t = rec[f"{kind}{j}"].view(-1, wh, ww, 90)
            img = ref_mod.window_reverse(t, (wh, ww), Hp, Wp)[:, :H, :W, :].contiguous()      # (B,H,W,90), crop of :696
            arrays[f"{kind}{j}"] = img.reshape(-1)[::S_STRIDE].numpy().copy()
        bias = probe_bias(scc)
        arrays[f"bias{j}_shape"] = np.array(bias.shape, dtype=np.int64)
        arrays[f"bias{j}"] = bias.reshape(-1)[::B_STRIDE].numpy().copy()
        print(f"block 0.{j}: window {wh} bias {tuple(bias.shape)} |bias|max {bias.abs().max():.4f}", flush=True)
    meta = dict(flags=list(flags), upsampler="nearest+conv", upscale=4, mode=mode, wseed=wseed, shape=list(shape), xseed=xseed,
                s_stride=S_STRIDE, b_stride=B_STRIDE)
    arrays["meta"] = np.array(repr(meta))
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **arrays)
    print(f"{name} -> {os.path.getsize(path) / 1e3:.0f} kB", flush=True)


def make_yardstick():
    """The reference's OWN bf16 error: the unmodified module under torch.autocast(bfloat16) against its fp32 run, for every golden case.
    north_star allows "bf16/fp32 compute" within a stated tolerance; this is the yardstick that tolerance is stated against
    (tests/helpers.py: the CUDA path may be at most 1.5x as far from the fp32 reference as the reference's own autocast run)."""
    import json
    import math
    sys.path.insert(0, HERE)
    from make_golden import CASES as SMALL
    cases = [(n, f, u, s, m, ws, sh, xs, 3) for (n, f, u, s, m, ws, sh, xs) in SMALL]
    cases += [(n, f, u, s, m, ws, sh, xs, 3) for (n, f, u, s, m, ws, sh, xs, _st, _c) in BIG]
    cases.append(("gray_x4_direct_40x44", (False, True, True), "pixelshuffledirect", 4, "stress", 15, (2, 40, 44), 25, 1))
    path = os.path.join(HERE, "bf16_yardstick.json")
    out = json.load(open(path)) if os.path.exists(path) else {}
    for name, flags, up, scale, mode, wseed, shape, xseed, ic in cases:
        if name in out:
            continue
        m, _ = build(flags, up, scale, mode, wseed, in_chans=ic)
        x = synthetic_image(*shape, seed=xseed, chans=ic)
        with torch.no_grad():
            y = m(x)
            with torch.autocast("cpu", dtype=torch.bfloat16):
                yb = m(x).float()
        scale_ = max(1.0, y.abs().max().item())
        err = (y - yb).abs().max().item() / scale_
        mse = (((y - yb) / scale_).double() ** 2).mean().item()
        out[name] = {"max_abs": err, "psnr": 10.0 * math.log10(1.0 / mse), "mode": mode, "shape": list(shape)}
        print(name, out[name], flush=True)
        json.dump(out, open(path, "w"), indent=1)


if __name__ == "__main__":
    what = sys.argv[1:] or ["small", "scc", "big"]
    if "yardstick" in what:
        make_yardstick()
    if "variants" in what:
        make_variants()
    if "small" in what:
        make_small()
    if "scc" in what:
        make_scc()
    if "big" in what:
        make_big()
