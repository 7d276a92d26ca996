"""Drop-in `HiT_SIR` for /root/reference/models/hit_sir_pro.py:1065-1344.

Same constructor signature (hit_sir_pro.py:1091-1120), same registered parameter tree and
state_dict keys (1650 for the "pro" configuration, no buffers), same `forward(x)` contract
(x: (B, in_chans, H>=33, W>=33) -> (B, in_chans, H*upscale, W*upscale)).  The modules below only
*hold parameters* under the reference's names; no arithmetic of the forward pass happens in
PyTorch -- `forward` hands raw device pointers to the C ABI (`include/hitsir_b200.h`).

Constructor variants built (SURVEY.md 8f-4): all four upsamplers incl. `upsampler=None` (denoise mode), `resi_connection` '1conv' and
'3conv', `ape=True`, `in_chans` 1 or 3, the three feature flags.  Not provided (SURVEY.md 8b): autograd/backward, widths other than
the pro width (embed_dim=180, 6 heads, mlp_ratio=2), `patch_norm=False`, dropout/drop-path > 0 in training mode; they raise
NotImplementedError where they would change the result.
"""
from __future__ import annotations

import contextlib
import ctypes
import math
import warnings
import weakref
from typing import Dict, Optional

import torch
import torch.nn as nn

try:  # the reference mixes this in (hit_sir_pro.py:9,1065); keep `from_pretrained`/`save_pretrained` working
    from huggingface_hub import PyTorchModelHubMixin
except Exception:  # pragma: no cover - huggingface_hub is present in the target image
    class PyTorchModelHubMixin:  # type: ignore
        pass

from . import _capi

# main.py:26-32 / test_experiment.py:25-32 of the reference: the "pro" configuration
PRO_KWARGS = dict(embed_dim=180, base_win_size=[8, 8], depths=[6] * 6, num_heads=[6] * 6, mlp_ratio=2,
                  upsampler="nearest+conv", hier_win_ratios=[0.5, 1, 2, 4, 6, 8, 10, 12])


# forward_x8 runs `group` of the eight dihedral transforms as one batch of group*B images.  A larger group means fewer, larger forwards
# (the forward is launch-bound at small sizes); past the size at which one forward fills the GPU it only costs workspace.  Largest
# group*B*H*W (LR pixels of one batched forward) a group may reach: the group sweep of DESIGN.md section 7.
X8_GROUP_TOKENS = 2_097_152


def x8_group(B: int, H: int, W: int) -> int:
    """Number of transforms forward_x8 batches together for a (B, *, H, W) input: the largest of 8 (square inputs only: the group
    holds both orientations), 4, 2 with group*B*H*W <= X8_GROUP_TOKENS and within the library's group*B*H*W*16 < 2^31, else 1."""
    for g in ((8, 4, 2) if H == W else (4, 2)):
        n = g * B * H * W
        if n <= X8_GROUP_TOKENS and n * 16 < 2 ** 31:
            return g
    return 1


def _ws_alloc_bytes(nbytes: int) -> int:
    """Size of a tensor that holds a library workspace of `nbytes` from its first 256-byte boundary on (_ws_offset)."""
    return nbytes + 256


def _ws_offset(ws: torch.Tensor) -> int:
    """Bytes from the start of `ws` to its first 256-byte boundary: the library takes 256-byte aligned workspaces."""
    return -ws.data_ptr() % 256


def _trunc_normal_(t: torch.Tensor, std: float = .02):
    # utils/arch_util.py:138-199 == timm trunc_normal_ (a=-2, b=2 in absolute units)
    return nn.init.trunc_normal_(t, mean=0., std=std, a=-2., b=2.)


def _destroy_handles(handles: dict) -> None:
    try:
        lib = _capi.load()
        for h in handles.values():
            lib.hitsir_destroy(h)
    except Exception:
        pass
    handles.clear()


class _NativeState:
    """Everything the module owns on the native side (C handles with their packed weights, the sync key, the cached workspace).
    It is not part of the module's value: `copy.deepcopy(model)` and pickling (`torch.save(model)`, EMA copies, DataLoader workers)
    give the copy a fresh, empty state that is re-created lazily on its first forward, exactly like a reference module that carries
    no native state at all.  Shallow replicas (`nn.DataParallel.replicate`, `copy.copy`) share this object; the handles are released
    when the LAST module referring to it is collected (weakref.finalize on the state object, not `__del__` on the module)."""

    def __init__(self):
        self.handles: Dict[int, ctypes.c_void_p] = {}
        self.synced: Dict[int, tuple] = {}
        self.workspaces: Dict[tuple, torch.Tensor] = {}
        self.params = None                      # cached parameter list for the cheap weights key
        weakref.finalize(self, _destroy_handles, self.handles)

    def __deepcopy__(self, memo):
        return _NativeState()

    def __reduce__(self):
        return (_NativeState, ())


# ----------------------------------------------------------------------------------------------
# parameter containers: names and shapes follow the reference classes line by line
# ----------------------------------------------------------------------------------------------
class _Holder(nn.Module):
    def forward(self, *a, **k):  # pragma: no cover
        raise RuntimeError("parameter container: the forward pass runs in the CUDA library")


class dwconv(_Holder):                      # hit_sir_pro.py:12-18
    def __init__(self, hidden_features):
        super().__init__()
        self.depthwise_conv = nn.Sequential(
            nn.Conv2d(hidden_features, hidden_features, kernel_size=5, stride=1, padding=2, dilation=1, groups=hidden_features),
            nn.GELU())


class ConvFFN(_Holder):                     # hit_sir_pro.py:27-37
    def __init__(self, in_features, hidden_features):
        super().__init__()
        self.fc1 = nn.Linear(in_features, hidden_features)
        self.dwconv = dwconv(hidden_features)
        self.fc2 = nn.Linear(hidden_features, in_features)


class MultipleSizeConvExtract(_Holder):     # hit_sir_pro.py:49-65
    def __init__(self, in_channels=3, out_channels=64):
        super().__init__()
        self.conv3 = nn.Conv2d(in_channels, out_channels, 3, 1, 1)
        self.conv5 = nn.Conv2d(in_channels, out_channels, 5, 1, 2)
        self.conv7 = nn.Conv2d(in_channels, out_channels, 7, 1, 3)
        self.conv9 = nn.Conv2d(in_channels, out_channels, 9, 1, 4)
        self.conv_x = nn.Conv2d(3, out_channels, 1, 1, 0)
        self.norm = nn.LayerNorm(out_channels)      # a state_dict key, never applied (:62)
        self.conv_last = nn.Conv2d(4 * out_channels, out_channels, 1, 1, 0)


class UnionAttention(_Holder):              # hit_sir_pro.py:104-111
    def __init__(self, in_channels):
        super().__init__()
        self.conv1 = nn.Conv2d(2, 1, 3, 1, 1)
        self.conv2 = nn.Conv2d(2, 1, 3, 1, 1)
        self.conv3 = nn.Conv2d(2, 1, 3, 1, 1)
        self.conv_last = nn.Conv2d(in_channels, in_channels, 3, 1, 1)


class Fusion(_Holder):                      # hit_sir_pro.py:136-143
    def __init__(self, out_channels=64):
        super().__init__()
        self.union_attention1 = UnionAttention(out_channels)
        self.union_attention2 = UnionAttention(out_channels)
        self.union_attention3 = UnionAttention(out_channels)


class DynamicPosBias(_Holder):              # hit_sir_pro.py:274-303
    def __init__(self, dim, num_heads):
        super().__init__()
        pos_dim = dim // 4
        self.pos_proj = nn.Linear(2, pos_dim)
        self.pos1 = nn.Sequential(nn.LayerNorm(pos_dim), nn.ReLU(inplace=True), nn.Linear(pos_dim, pos_dim))
        self.pos2 = nn.Sequential(nn.LayerNorm(pos_dim), nn.ReLU(inplace=True), nn.Linear(pos_dim, pos_dim))
        self.pos3 = nn.Sequential(nn.LayerNorm(pos_dim), nn.ReLU(inplace=True), nn.Linear(pos_dim, num_heads))


class SpatialChannelAttention(_Holder):     # hit_sir_pro.py:317-336
    def __init__(self, dim):
        super().__init__()
        self.linear1 = nn.Conv2d(1, dim, 3, 1, 1)
        self.linear2 = nn.Conv2d(1, dim, 3, 1, 1)
        self.linear1_first = nn.Linear(dim, dim // 10)
        self.linear1_second = nn.Linear(dim // 10, dim)
        self.linear2_first = nn.Linear(dim, dim // 10)
        self.linear2_second = nn.Linear(dim // 10, dim)


class SCC(_Holder):                         # hit_sir_pro.py:362-433
    def __init__(self, is_channel_spatial_attn, dim, base_win_size, window_size, num_heads):
        super().__init__()
        self.qkv = SpatialChannelAttention(dim) if is_channel_spatial_attn else nn.Identity()
        self.proj = nn.Linear(dim, dim)
        base = (min(window_size[0], base_win_size[0]), min(window_size[1], base_win_size[1]))
        head_dim = dim // (2 * num_heads)
        self.spatial_linear = nn.Linear((window_size[0] * window_size[1]) // (base[0] * base[1]), 1)
        self.k_generate1 = nn.Linear(head_dim, head_dim)
        self.k_generate2 = nn.Linear(head_dim, head_dim)
        self.pos = DynamicPosBias(dim // 4, num_heads)


class HierarchicalTransformerBlock(_Holder):   # hit_sir_pro.py:605-662
    def __init__(self, is_channel_spatial_attn, dim, num_heads, base_win_size, window_size, mlp_ratio):
        super().__init__()
        if window_size[0] > base_win_size[0] and window_size[1] > base_win_size[1]:
            assert window_size[0] % base_win_size[0] == 0, "please ensure the window size is smaller than or divisible by the base window size"
            assert window_size[1] % base_win_size[1] == 0, "please ensure the window size is smaller than or divisible by the base window size"
        self.norm1 = nn.LayerNorm(dim)
        self.correlation = SCC(is_channel_spatial_attn, dim, base_win_size, window_size, num_heads)
        self.norm2 = nn.LayerNorm(dim)
        self.mlp = ConvFFN(dim, int(dim * mlp_ratio))


class BasicLayer(_Holder):                  # hit_sir_pro.py:755-823
    def __init__(self, is_channel_spatial_attn, dim, depth, num_heads, base_win_size, mlp_ratio, hier_win_ratios):
        super().__init__()
        win_hs = [int(base_win_size[0] * r) for r in hier_win_ratios]
        win_ws = [int(base_win_size[1] * r) for r in hier_win_ratios]
        self.blocks = nn.ModuleList([
            HierarchicalTransformerBlock(is_channel_spatial_attn, dim, num_heads, base_win_size, (win_hs[i], win_ws[i]), mlp_ratio)
            for i in range(depth)])


def _resi_conv(dim, resi_connection):        # hit_sir_pro.py:911-918, 1221-1231
    if resi_connection == '1conv':
        return nn.Conv2d(dim, dim, 3, 1, 1)
    return nn.Sequential(nn.Conv2d(dim, dim // 4, 3, 1, 1), nn.LeakyReLU(negative_slope=0.2, inplace=True),
                         nn.Conv2d(dim // 4, dim // 4, 1, 1, 0), nn.LeakyReLU(negative_slope=0.2, inplace=True),
                         nn.Conv2d(dim // 4, dim, 3, 1, 1))


class RHTB(_Holder):                        # hit_sir_pro.py:848-926
    def __init__(self, is_channel_spatial_attn, dim, depth, num_heads, base_win_size, mlp_ratio, hier_win_ratios, resi_connection='1conv'):
        super().__init__()
        self.residual_group = BasicLayer(is_channel_spatial_attn, dim, depth, num_heads, base_win_size, mlp_ratio, hier_win_ratios)
        self.conv = _resi_conv(dim, resi_connection)


class PatchEmbed(_Holder):                  # hit_sir_pro.py:939-973
    def __init__(self, embed_dim, norm_layer=None):
        super().__init__()
        self.norm = norm_layer(embed_dim) if norm_layer is not None else None


class Upsample(nn.Sequential):              # hit_sir_pro.py:1024-1043
    def __init__(self, scale, num_feat):
        m = []
        if (scale & (scale - 1)) == 0:
            for _ in range(int(math.log(scale, 2))):
                m.append(nn.Conv2d(num_feat, 4 * num_feat, 3, 1, 1))
                m.append(nn.PixelShuffle(2))
        elif scale == 3:
            m.append(nn.Conv2d(num_feat, 9 * num_feat, 3, 1, 1))
            m.append(nn.PixelShuffle(3))
        else:
            raise ValueError(f'scale {scale} is not supported. ' 'Supported scales: 2^n and 3.')
        super().__init__(*m)


class UpsampleOneStep(nn.Sequential):       # hit_sir_pro.py:1046-1062
    def __init__(self, scale, num_feat, num_out_ch):
        super().__init__(nn.Conv2d(num_feat, (scale ** 2) * num_out_ch, 3, 1, 1), nn.PixelShuffle(scale))


# ----------------------------------------------------------------------------------------------
class HiT_SIR(nn.Module, PyTorchModelHubMixin):
    """HiT-SIR network; constructor mirrors hit_sir_pro.py:1091-1120 argument for argument."""

    def __init__(self,
                 is_mult_size_conv_feat_extract: bool,
                 is_channel_spatial_attn: bool,
                 is_fusion: bool,
                 img_size=64, patch_size=1, in_chans=3, embed_dim=60,
                 depths=[6, 6, 6, 6], num_heads=[6, 6, 6, 6], base_win_size=[8, 8], mlp_ratio=2.,
                 drop_rate=0., value_drop_rate=0., drop_path_rate=0.,
                 norm_layer=nn.LayerNorm, ape=False, patch_norm=True, use_checkpoint=False,
                 upscale=4, img_range=1., upsampler='pixelshuffledirect', resi_connection='1conv',
                 hier_win_ratios=[0.5, 1, 2, 4, 6, 8], **kwargs):
        super().__init__()
        depths, num_heads = list(depths), list(num_heads)
        base_win_size, hier_win_ratios = list(base_win_size), list(hier_win_ratios)
        num_feat = 64
        self.img_range = img_range
        if in_chans == 3:
            self.mean = torch.Tensor((0.485, 0.456, 0.4060)).view(1, 3, 1, 1)   # plain attribute, not a buffer (:1128-1129)
        else:
            self.mean = torch.zeros(1, 1, 1, 1)
        self.upscale, self.upsampler, self.base_win_size = upscale, upsampler, base_win_size
        self.num_layers, self.embed_dim, self.ape, self.patch_norm = len(depths), embed_dim, ape, patch_norm
        self.num_features, self.mlp_ratio = embed_dim, mlp_ratio
        self.in_chans, self.depths, self.num_heads, self.hier_win_ratios = in_chans, depths, num_heads, hier_win_ratios
        self.flags = (bool(is_mult_size_conv_feat_extract), bool(is_channel_spatial_attn), bool(is_fusion))
        self.drop_rates = (drop_rate, value_drop_rate, drop_path_rate)

        # what this build cannot compute is refused up front (nothing silently differs from the reference)
        if norm_layer is not nn.LayerNorm:
            raise NotImplementedError("hitsir_b200: only norm_layer=nn.LayerNorm")
        if not patch_norm:
            raise NotImplementedError("hitsir_b200: patch_norm=False is not implemented")
        if resi_connection not in ('1conv', '3conv'):
            raise NotImplementedError(f"hitsir_b200: resi_connection={resi_connection!r} is not implemented")
        if upsampler == 'pixelshuffle' and (upscale & (upscale - 1)) == 0 and upscale > 4:
            raise NotImplementedError(f"hitsir_b200: upsampler='pixelshuffle' with upscale={upscale} is not implemented (1, 2, 3, 4)")
        if embed_dim != 180 or any(h != 6 for h in num_heads) or float(mlp_ratio) != 2.0:
            raise NotImplementedError("hitsir_b200 implements the HiT-SIR-pro width: embed_dim=180, num_heads=6, mlp_ratio=2 "
                                      f"(got embed_dim={embed_dim}, num_heads={num_heads}, mlp_ratio={mlp_ratio})")
        if upsampler not in ('pixelshuffle', 'pixelshuffledirect', 'nearest+conv', None, ''):
            raise NotImplementedError(f"hitsir_b200: upsampler={upsampler!r} is not implemented")
        self.resi_connection = resi_connection
        self.img_size, self.patch_size = img_size, patch_size
        if ape:                                  # direct parameter of the top module: first key of the state_dict, like the reference (:1187-1189)
            n = img_size if isinstance(img_size, (tuple, list)) else (img_size, img_size)
            ps = patch_size if isinstance(patch_size, (tuple, list)) else (patch_size, patch_size)
            self.absolute_pos_embed = nn.Parameter(torch.zeros(1, (n[0] // ps[0]) * (n[1] // ps[1]), embed_dim))
            _trunc_normal_(self.absolute_pos_embed, std=.02)

        # 1. shallow feature extraction (:1139-1154)
        if is_mult_size_conv_feat_extract:
            self.conv_first = MultipleSizeConvExtract(in_chans, embed_dim)
        else:
            self.conv_first = nn.Conv2d(in_chans, embed_dim, 3, 1, 1)
        self.fusion = Fusion(embed_dim) if is_fusion else (lambda x, y: x + y)
        # 2. deep feature extraction (:1158-1231)
        self.patch_embed = PatchEmbed(embed_dim, norm_layer if patch_norm else None)
        self.layers = nn.ModuleList([
            RHTB(is_channel_spatial_attn, embed_dim, depths[i], num_heads[i], base_win_size, mlp_ratio, hier_win_ratios, resi_connection)
            for i in range(self.num_layers)])
        self.norm = norm_layer(embed_dim)
        self.conv_after_body = _resi_conv(embed_dim, resi_connection)
        # 3. reconstruction (:1235-1262)
        if upsampler == 'pixelshuffle':
            self.conv_before_upsample = nn.Sequential(nn.Conv2d(embed_dim, num_feat, 3, 1, 1), nn.LeakyReLU(inplace=True))
            self.upsample = Upsample(upscale, num_feat)
            self.conv_last = nn.Conv2d(num_feat, in_chans, 3, 1, 1)
        elif upsampler == 'pixelshuffledirect':
            self.upsample = UpsampleOneStep(upscale, embed_dim, in_chans)
        elif upsampler == 'nearest+conv':
            assert self.upscale == 4, 'only support x4 now.'
            self.conv_before_upsample = nn.Sequential(nn.Conv2d(embed_dim, num_feat, 3, 1, 1), nn.LeakyReLU(inplace=True))
            self.conv_up1 = nn.Conv2d(num_feat, num_feat, 3, 1, 1)
            self.conv_up2 = nn.Conv2d(num_feat, num_feat, 3, 1, 1)
            self.conv_hr = nn.Conv2d(num_feat, num_feat, 3, 1, 1)
            self.conv_last = nn.Conv2d(num_feat, in_chans, 3, 1, 1)
        else:                                    # denoising / compression-artefact mode (:1260-1262): x + conv_last(res)
            self.conv_last = nn.Conv2d(embed_dim, in_chans, 3, 1, 1)
        self.apply(self._init_weights)

        # native state (never part of state_dict, never copied or pickled: see _NativeState)
        self._native = _NativeState()
        self._forced_workspace: Optional[torch.Tensor] = None      # set by GraphedForward around its capture
        self._inject_src: Optional[torch.Tensor] = None
        self._warned_grad = False
        self.last_launch_count = 0

    def _init_weights(self, m):                 # hit_sir_pro.py:1267-1274
        if isinstance(m, nn.Linear):
            _trunc_normal_(m.weight, std=.02)
            if m.bias is not None:
                nn.init.constant_(m.bias, 0)
        elif isinstance(m, nn.LayerNorm):
            nn.init.constant_(m.bias, 0)
            nn.init.constant_(m.weight, 1.0)

    @torch.jit.ignore
    def no_weight_decay(self):
        return {'absolute_pos_embed'}

    @torch.jit.ignore
    def no_weight_decay_keywords(self):
        return {'relative_position_bias_table'}

    # ------------------------------------------------------------------ native plumbing
    def _config(self) -> _capi.HitsirConfig:
        c = _capi.HitsirConfig()
        c.is_mult_size_conv_feat_extract, c.is_channel_spatial_attn, c.is_fusion = [int(f) for f in self.flags]
        c.in_chans, c.embed_dim, c.num_layers = self.in_chans, self.embed_dim, self.num_layers
        if self.num_layers > _capi.HITSIR_MAX_LAYERS or len(self.hier_win_ratios) > _capi.HITSIR_MAX_DEPTH:
            raise NotImplementedError("hitsir_b200: at most 16 layers / 16 window ratios")
        for i in range(self.num_layers):
            c.depths[i], c.num_heads[i] = self.depths[i], self.num_heads[i]
        c.base_win_size[0], c.base_win_size[1] = self.base_win_size
        c.mlp_ratio, c.upscale, c.img_range = float(self.mlp_ratio), int(self.upscale), float(self.img_range)
        c.upsampler = _capi.UPSAMPLERS[self.upsampler]
        c.num_ratios = len(self.hier_win_ratios)
        for i, r in enumerate(self.hier_win_ratios):
            c.hier_win_ratios[i] = float(r)
        c.resi_3conv = 1 if self.resi_connection == '3conv' else 0
        c.ape_tokens = int(self.absolute_pos_embed.shape[1]) if self.ape else 0
        return c

    @property
    def out_scale(self) -> int:
        """Spatial factor of the output: `upscale`, except upsampler=None, whose forward returns x-sized images (:1340-1344)."""
        return self.upscale if self.upsampler else 1

    def _handle(self, device: torch.device) -> ctypes.c_void_p:
        idx = device.index if device.index is not None else torch.cuda.current_device()
        h = self._native.handles.get(idx)
        if h is None:
            lib = _capi.load()
            cfg = self._config()
            out = ctypes.c_void_p()
            with torch.cuda.device(idx):
                _capi.check(lib.hitsir_create(ctypes.byref(cfg), ctypes.byref(out)))
            h = out
            self._native.handles[idx] = h
            # the C side and this module must agree on the state_dict key set
            names = {lib.hitsir_param_name(h, i).decode() for i in range(lib.hitsir_num_params(h))}
            mine = set(self.state_dict().keys())
            if names != mine:
                raise RuntimeError(f"hitsir_b200: parameter registry mismatch: only-native={sorted(names - mine)[:5]} "
                                   f"only-python={sorted(mine - names)[:5]}")
        return h

    def _weights_key(self):
        # in-place updates (optimizer steps, load_state_dict's copy_) bump Tensor._version; the parameter list itself is cached
        # because walking the 1650-entry module tree costs more than a small forward (invalidated by _apply / refresh_weights)
        ns = self._native
        if ns.params is None:
            ns.params = list(self.parameters())
        return tuple([p._version for p in ns.params])

    def refresh_weights(self):
        """Force re-packing on the next forward (needed only after `param.data = ...` style rebinding or after replacing a
        Parameter object)."""
        self._native.synced.clear()
        self._native.params = None

    def _apply(self, fn, *args, **kwargs):      # .to() / .cuda() / .float() ... move storage: re-pack
        self._native.synced.clear()
        self._native.params = None
        return super()._apply(fn, *args, **kwargs)

    def load_state_dict(self, *args, **kwargs):
        self._native.params = None
        return super().load_state_dict(*args, **kwargs)

    def _sync_weights(self, h, device: torch.device, stream: int):
        idx = device.index if device.index is not None else torch.cuda.current_device()
        key = self._weights_key()
        if self._native.synced.get(idx) == key:
            return
        lib = _capi.load()
        keep = []
        for name, p in self.state_dict(keep_vars=True).items():
            t = p.detach()
            if t.device != device or t.dtype != torch.float32 or not t.is_contiguous():
                t = t.to(device=device, dtype=torch.float32).contiguous()
                keep.append(t)
            _capi.check(lib.hitsir_set_param(h, name.encode(), ctypes.c_void_p(t.data_ptr()), t.numel(), ctypes.c_void_p(stream)))
        _capi.check(lib.hitsir_finalize_weights(h, ctypes.c_void_p(stream)))
        self._native.synced[idx] = key
        del keep

    def _workspace(self, h, device, B, H, W, group=0) -> torch.Tensor:
        key = (device.index, B, H, W, group)
        ws = self._native.workspaces.get(key)
        if ws is None:
            # one live workspace per kind (forward: group 0, forward_x8: group > 0): shapes rarely alternate, and alternating
            # forward / forward_x8 calls keep both
            for k in [k for k in self._native.workspaces if (k[4] > 0) == (group > 0)]:
                del self._native.workspaces[k]
            ws = self.new_workspace(device, B, H, W, group)
            self._native.workspaces[key] = ws
        return ws

    def new_workspace(self, device, B, H, W, group=0) -> torch.Tensor:
        """A scratch buffer for a (B,H,W) forward that the caller owns (GraphedForward keeps one per captured graph, so that
        neither a forward with another shape nor a weight update can free memory a captured launch still points to).
        group > 0: the buffer of forward_x8 with that group (hitsir_workspace_bytes_x8)."""
        device = torch.device(device)
        n = ctypes.c_size_t()
        with torch.cuda.device(device):
            lib, h = _capi.load(), self._handle(device)
            if group:
                _capi.check(lib.hitsir_workspace_bytes_x8(h, B, H, W, group, ctypes.byref(n)))
            else:
                _capi.check(lib.hitsir_workspace_bytes(h, B, H, W, ctypes.byref(n)))
        return torch.empty(_ws_alloc_bytes(n.value), dtype=torch.uint8, device=device)

    @contextlib.contextmanager
    def _native_call(self, device, shape=None, ws: Optional[torch.Tensor] = None, stream: Optional[int] = None):
        """Enters `device` for one call of a forward entry of the C ABI: creates the handle and syncs the weights on `stream` (default:
        the device's current stream), then yields (library, handle, workspace pointer, workspace bytes, stream) for `ws`, or for the
        cached workspace of `shape` = (B, H, W[, group]) when `ws` is None."""
        with torch.cuda.device(device):
            stream = torch.cuda.current_stream(device).cuda_stream if stream is None else stream
            h = self._handle(device)
            self._sync_weights(h, device, stream)
            if ws is None:
                ws = self._workspace(h, device, *shape)
            off = _ws_offset(ws)
            yield _capi.load(), h, ctypes.c_void_p(ws.data_ptr() + off), ws.numel() - off, ctypes.c_void_p(stream)

    def set_inject(self, device, name: Optional[str], src: Optional[torch.Tensor] = None):
        """Test hook (stands in for a forward pre-hook that replaces a sub-module's input), see hitsir_set_inject.  `src` is kept
        alive by the module until cleared."""
        h = self._handle(torch.device(device))
        if name is None:
            self._inject_src = None
            _capi.check(_capi.load().hitsir_set_inject(h, None, None, 0))
        else:
            src = src.detach().to(device=device, dtype=torch.float32).contiguous()
            self._inject_src = src
            _capi.check(_capi.load().hitsir_set_inject(h, name.encode(), ctypes.c_void_p(src.data_ptr()), src.numel()))

    def bias_table(self, device, layer: int, block: int) -> torch.Tensor:
        """The pooled relative-position bias (6, L, Lb) of block (layer, block) as the library precomputed it (hit_sir_pro.py:477-503)."""
        device = torch.device(device)
        win = int(self.base_win_size[0] * self.hier_win_ratios[block])
        base = min(win, self.base_win_size[0])
        out = torch.empty((6, win * win, base * base), dtype=torch.float32, device=device)
        with torch.cuda.device(device):
            stream = torch.cuda.current_stream(device).cuda_stream
            h = self._handle(device)
            self._sync_weights(h, device, stream)
            _capi.check(_capi.load().hitsir_get_bias_table(h, layer, block, ctypes.c_void_p(out.data_ptr()), out.numel(), ctypes.c_void_p(stream)))
        return out

    def set_tap(self, device, name: Optional[str], dst: Optional[torch.Tensor] = None, stop: bool = True):
        """Test hook (stands in for forward hooks on reference sub-modules), see hitsir_set_tap."""
        h = self._handle(torch.device(device))
        if name is None:
            _capi.check(_capi.load().hitsir_set_tap(h, None, None, 0, 0))
        else:
            _capi.check(_capi.load().hitsir_set_tap(h, name.encode(), ctypes.c_void_p(dst.data_ptr()), dst.numel(), int(stop)))

    def profile_enable(self, device, on: bool = True):
        """Per-category CUDA-event timing of the kernel launches (hitsir_profile_enable); resets the totals."""
        _capi.check(_capi.load().hitsir_profile_enable(self._handle(torch.device(device)), int(on)))

    def profile_read(self, device) -> Dict[str, tuple]:
        """{category: (total_ms, launches)} since profile_enable; synchronise the stream first."""
        lib = _capi.load()
        h = self._handle(torch.device(device))
        out = {}
        for i in range(lib.hitsir_profile_num_categories(h)):
            name, ms, n = ctypes.c_char_p(), ctypes.c_double(), ctypes.c_int64()
            _capi.check(lib.hitsir_profile_get(h, i, ctypes.byref(name), ctypes.byref(ms), ctypes.byref(n)))
            if n.value:
                out[name.value.decode()] = (ms.value, n.value)
        return out

    def set_gemm_backend(self, device, backend: str):
        _capi.check(_capi.load().hitsir_set_gemm_backend(self._handle(torch.device(device)), backend.encode()))

    # ------------------------------------------------------------------ forward
    def _check_input(self, x: torch.Tensor) -> None:
        if x.dim() != 4 or x.shape[1] != self.in_chans:
            raise RuntimeError(f"expected input of shape (B, {self.in_chans}, H, W), got {tuple(x.shape)}")
        if not x.is_cuda:
            raise RuntimeError("hitsir_b200.HiT_SIR runs on a CUDA (sm_100) device only: there is no CPU path. "
                               "Move the module and the input to 'cuda'.")
        if self.training and any(r > 0 for r in self.drop_rates):
            raise NotImplementedError("hitsir_b200: dropout / drop-path > 0 in training mode is not implemented")
        if torch.is_grad_enabled() and self.training and not self._warned_grad:
            warnings.warn("hitsir_b200.HiT_SIR computes the forward pass only; the result carries no autograd graph.")
            self._warned_grad = True
        self.mean = self.mean.type_as(x)        # same side effect as the reference (:1310)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        """x: (B, in_chans, H, W) on a CUDA device -> (B, in_chans, H*upscale, W*upscale).  hit_sir_pro.py:1304-1344."""
        self._check_input(x)
        B, _, H, W = x.shape
        in_dtype = x.dtype
        xin = x.detach().to(torch.float32).contiguous()
        y = torch.empty((B, self.in_chans, H * self.out_scale, W * self.out_scale), dtype=torch.float32, device=xin.device)
        with self._native_call(xin.device, (B, H, W), self._forced_workspace) as (lib, h, ws, ws_bytes, st):
            _capi.check(lib.hitsir_forward(h, ctypes.c_void_p(xin.data_ptr()), ctypes.c_void_p(y.data_ptr()), B, H, W, ws, ws_bytes, st))
            self.last_launch_count = int(lib.hitsir_last_launch_count(h))
        return y if in_dtype == torch.float32 else y.to(in_dtype)

    def forward_x8(self, x: torch.Tensor) -> torch.Tensor:
        """x8 geometric self-ensemble (the "+" mode of EDSR+ / RCAN+ / SwinIR+, BasicSR's test_selfensemble): the mean of
        T_k^-1(forward(T_k(x))) over the eight flips / transposes T_k, summed in ascending k in fp32 and scaled by 1/8 (hitsir_forward_x8).
        Same input contract, errors and output as `forward`; 8x its work, batched `x8_group(B, H, W)` transforms at a time."""
        return self._forward_x8(x, None)

    def _forward_x8(self, x: torch.Tensor, group: Optional[int]) -> torch.Tensor:
        self._check_input(x)
        B, _, H, W = x.shape
        group = x8_group(B, H, W) if group is None else group
        in_dtype = x.dtype
        xin = x.detach().to(torch.float32).contiguous()
        y = torch.empty((B, self.in_chans, H * self.out_scale, W * self.out_scale), dtype=torch.float32, device=xin.device)
        with self._native_call(xin.device, (B, H, W, group)) as (lib, h, ws, ws_bytes, st):
            _capi.check(lib.hitsir_forward_x8(h, ctypes.c_void_p(xin.data_ptr()), ctypes.c_void_p(y.data_ptr()), B, H, W, group,
                                              ws, ws_bytes, st))
            self.last_launch_count = int(lib.hitsir_last_launch_count(h))
        return y if in_dtype == torch.float32 else y.to(in_dtype)

    def forward_host(self, x_host: torch.Tensor, y_host: Optional[torch.Tensor] = None, device=None) -> torch.Tensor:
        """End-to-end call on HOST tensors through hitsir_forward_host (H2D copy, forward, D2H copy on the
        current stream; returns after a stream synchronize).  `x_host` should be pinned."""
        device = torch.device(device if device is not None else next(self.parameters()).device)
        if device.type != "cuda":
            raise RuntimeError("hitsir_b200.HiT_SIR runs on a CUDA (sm_100) device only: there is no CPU path.")
        B, _, H, W = x_host.shape
        x_host = x_host.contiguous().float()
        if y_host is None:
            y_host = torch.empty((B, self.in_chans, H * self.out_scale, W * self.out_scale), dtype=torch.float32, pin_memory=True)
        dx = torch.empty(x_host.shape, dtype=torch.float32, device=device)
        dy = torch.empty(y_host.shape, dtype=torch.float32, device=device)
        with self._native_call(device, (B, H, W)) as (lib, h, ws, ws_bytes, st):
            _capi.check(lib.hitsir_forward_host(h, ctypes.c_void_p(x_host.data_ptr()), ctypes.c_void_p(y_host.data_ptr()), B, H, W,
                                                ctypes.c_void_p(dx.data_ptr()), ctypes.c_void_p(dy.data_ptr()), ws, ws_bytes, st))
            torch.cuda.current_stream(device).synchronize()
            self.last_launch_count = int(lib.hitsir_last_launch_count(h))
        return y_host

    def forward_uint8(self, x_u8: torch.Tensor, self_ensemble: bool = False) -> torch.Tensor:
        """PIL-style images in, PIL-style images out, without leaving the device: `x_u8` (B,H,W,C) uint8 CUDA tensor ->
        (B, sH, sW, C) uint8 = to_pil_image(model(to_tensor(x)).clip(0, 1)) of test_experiment.py:70-77 (utils/utils.py:143-145,
        experiments/experiment.py:746-748).  The D2H copy of the result is 4x smaller than the fp32 NCHW output.
        self_ensemble=True: the same round trip around forward_x8 (hitsir_forward_x8_u8), bit-identical to
        to_uint8_hwc(forward_x8(to_tensor(x)))."""
        if x_u8.device.type != "cuda" or x_u8.dtype != torch.uint8 or x_u8.dim() != 4:
            raise RuntimeError("forward_uint8 expects a (B,H,W,C) uint8 CUDA tensor: there is no CPU path.")
        B, H, W, C = x_u8.shape
        if C != self.in_chans:
            raise RuntimeError(f"expected {self.in_chans} channels, got {C}")
        device = x_u8.device
        x_u8 = x_u8.contiguous()
        y = torch.empty((B, H * self.out_scale, W * self.out_scale, C), dtype=torch.uint8, device=device)
        if self_ensemble:
            group = x8_group(B, H, W)
            with self._native_call(device, (B, H, W, group)) as (lib, h, ws, ws_bytes, st):
                _capi.check(lib.hitsir_forward_x8_u8(h, ctypes.c_void_p(x_u8.data_ptr()), ctypes.c_void_p(y.data_ptr()), B, H, W, group,
                                                     ws, ws_bytes, st))
                self.last_launch_count = int(lib.hitsir_last_launch_count(h))
            return y
        dx = torch.empty((B, C, H, W), dtype=torch.float32, device=device)
        dy = torch.empty((B, C, H * self.out_scale, W * self.out_scale), dtype=torch.float32, device=device)
        with self._native_call(device, (B, H, W)) as (lib, h, ws, ws_bytes, st):
            _capi.check(lib.hitsir_forward_u8(h, ctypes.c_void_p(x_u8.data_ptr()), ctypes.c_void_p(y.data_ptr()), B, H, W,
                                              ctypes.c_void_p(dx.data_ptr()), ctypes.c_void_p(dy.data_ptr()), ws, ws_bytes, st))
            self.last_launch_count = int(lib.hitsir_last_launch_count(h))
        return y

    def load_checkpoint(self, path_or_dict, map_location="cpu") -> Optional[int]:
        """Load a checkpoint written by the reference harness (experiments/experiment.py:257-263: {'start_epoch', 'model',
        'optimizer'}; read back at :222-223 and test_experiment.py:43-44) or a bare state_dict, strictly.  Returns
        'start_epoch' when present."""
        ck = path_or_dict if isinstance(path_or_dict, dict) else torch.load(path_or_dict, map_location=map_location, weights_only=True)
        sd = ck["model"] if isinstance(ck, dict) and "model" in ck and isinstance(ck["model"], dict) else ck
        self.load_state_dict(sd, strict=True)
        return ck.get("start_epoch") if isinstance(ck, dict) and "start_epoch" in ck else None

    def native_handle(self, device) -> int:
        """Address of the C handle bound to `device` (None before the first forward there): GraphedForward uses it to notice that the
        handle a captured graph points into has been replaced."""
        idx = torch.device(device).index
        h = self._native.handles.get(idx if idx is not None else torch.cuda.current_device())
        return None if h is None else h.value
