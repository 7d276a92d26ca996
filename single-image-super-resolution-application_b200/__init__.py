"""hitsir_b200 -- B200-native (sm_100a) implementation of the HiT-SIR-pro forward pass.

Host-side mirror of the reference interface for ONE path:
`models/hit_sir_pro.py::HiT_SIR` of CoderLinxin/Single-Image-Super-Resolution-Application.
`HiT_SIR` here is a drop-in `torch.nn.Module` (same constructor, same state_dict keys, same
`forward(x)` contract); the arithmetic runs in hand-written CUDA kernels behind the C ABI of
`include/hitsir_b200.h` (tcgen05/TMEM/TMA contractions + fused glue kernels).  PyTorch only
provides device memory, streams and `torch.distributed` plumbing.
"""
from .hit_sir_pro import HiT_SIR, PRO_KWARGS  # noqa: F401
from . import _capi  # noqa: F401
from .sharding import ShardedSR, PeerGather, tile_plan, stitch_tiles  # noqa: F401
from .host_pipeline import HostPipeline  # noqa: F401
from .metrics import mse_y, psnr_y, ssim_y, psnr_ssim_basicsr, to_uint8_hwc  # noqa: F401
from .resize import resize_bicubic, to_float_nchw, evaluate  # noqa: F401
from .graphed import GraphedForward  # noqa: F401
from .banded import BandedSR, LocalBandedSR, band_plan  # noqa: F401

__all__ = ["HiT_SIR", "PRO_KWARGS", "ShardedSR", "tile_plan", "stitch_tiles", "HostPipeline", "mse_y", "psnr_y", "ssim_y", "psnr_ssim_basicsr", "to_uint8_hwc", "resize_bicubic", "to_float_nchw", "evaluate", "GraphedForward", "BandedSR", "LocalBandedSR", "band_plan", "PeerGather"]
