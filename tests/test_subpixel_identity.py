"""The identity behind `conv3_c64_up_kernel` / `pack_subpixel_kernel` (csrc/conv3_c64.cu, csrc/pack.cu): a 3x3 conv of a x2
nearest-upsampled map (/root/reference/models/hit_sir_pro.py:1331-1332) equals four 2x2 convs of the map itself, one per output phase,
whose filters are sums of the 3x3 taps that land on the same source pixel.  CPU only; the GPU taps `up1` / `up2` check the kernel."""
import torch
import torch.nn.functional as F

# taps of the 3x3 filter that fall on LR offset index 0 / 1 for output phase bit 0 / 1 (same table as pack_subpixel_kernel)
TAPS = {(0, 0): (0,), (0, 1): (1, 2), (1, 0): (0, 1), (1, 1): (2,)}


def phase_filter(w, a, bb, dyi, dxi):
    """The (Co, Ci) filter of output phase (a, bb) at LR offset index (dyi, dxi): its taps summed in pack_subpixel_kernel's order."""
    return sum(w[:, :, ky, kx] for ky in TAPS[(a, dyi)] for kx in TAPS[(bb, dxi)])


def subpixel_conv(x, w, b, filt=phase_filter):
    n, _, h, wd = x.shape
    out = torch.empty(n, w.shape[0], 2 * h, 2 * wd, dtype=x.dtype)
    xp = F.pad(x, (1, 1, 1, 1))
    for a in range(2):
        for bb in range(2):
            acc = b.view(1, -1, 1, 1).expand(n, -1, h, wd).clone()
            for dyi in range(2):
                for dxi in range(2):
                    wp = filt(w, a, bb, dyi, dxi)
                    dy, dx = a - 1 + dyi, bb - 1 + dxi
                    acc = acc + torch.einsum("oc,nchw->nohw", wp, xp[:, :, 1 + dy:1 + dy + h, 1 + dx:1 + dx + wd])
            out[:, :, a::2, bb::2] = acc
    return out


def test_subpixel_filters_equal_conv_of_nearest_upsampled_map():
    g = torch.Generator().manual_seed(3)
    for (h, w) in ((7, 9), (1, 1), (8, 16), (33, 5)):
        x = torch.randn(2, 5, h, w, generator=g, dtype=torch.float64)
        wt = torch.randn(6, 5, 3, 3, generator=g, dtype=torch.float64)
        b = torch.randn(6, generator=g, dtype=torch.float64)
        ref = F.conv2d(F.interpolate(x, scale_factor=2, mode="nearest"), wt, b, 1, 1)
        assert torch.allclose(subpixel_conv(x, wt, b), ref, rtol=0, atol=1e-12)


def test_identity_filter_stays_exact():
    """a centre-tap identity conv is still an exact copy in phase form (the bit-exact nearest test relies on it)"""
    x = torch.randn(1, 4, 6, 6, dtype=torch.float64)
    wt = torch.zeros(4, 4, 3, 3, dtype=torch.float64)
    for c in range(4):
        wt[c, c, 1, 1] = 1.0
    got = subpixel_conv(x, wt, torch.zeros(4, dtype=torch.float64))
    assert torch.equal(got, F.interpolate(x, scale_factor=2, mode="nearest"))
