"""Timing of BasicSR's PSNR / SSIM on the device (hitsir_b200.psnr_ssim_basicsr) and of the tensor2img rounding conversion.

    python tools/bench_basicsr_metrics.py [--steps K] [--warmup W] [--window S]

Prints ONE JSON line with, per size, ms per call of psnr_ssim_basicsr in Y mode (test_y_channel=True) and RGB mode, crop_border 4,
on uint8 (B,H,W,3) batches; ms of to_uint8_hwc(rounding="nearest") at cfg2's output; each as a fraction of one cfg2 forward
(32x3x256x256 LR, x4, pro configuration); and the CPU time of the cv2/numpy restatement of BasicSR (tests/basicsr_ref.py) on the
DIV2K image.  Sizes:
  "div2k":  one DIV2K validation HR image, 1x1356x2040x3.  A pair is 17 MB, so the calls rotate over 10 pairs (166 MB, more than the
            126 MB L2);
  "cfg2":   cfg2's output, 32x1024x1024x3 (201 MB per pair, larger than L2 by itself);
  "cfg1":   cfg1's output, 1x256x256x3 (L2-resident and launch-bound: a measure of overheads).
GB/s counts 6 algorithmic bytes per pixel (two uint8 RGB images read once).
Timed regions: profiling off, CUDA events on the current stream after a synchronize, at least K calls and at least --window seconds
after W warm-up calls.  The GPU name, power limit and SM clocks are read with nvidia-smi in the same run.
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from tools.bench_ssim import gpu_info, rotating, time_call  # noqa: E402

BYTES_PER_PIXEL = 6       # sr and hr, 3 uint8 channels each
SIZES = {"div2k": ((1, 1356, 2040), 10), "cfg2": ((32, 1024, 1024), 1), "cfg1": ((1, 256, 256), 1)}   # shape, rotated pairs
CROP = 4


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--window", type=float, default=1.0, help="least seconds per timed region")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_basicsr_metrics.py needs a CUDA device (B200)")
    import hitsir_b200

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    info = gpu_info(0)
    g = torch.Generator(device=dev)
    g.manual_seed(1234)
    res = {"metric": "psnr_ssim_basicsr ms per call", "crop_border": CROP, "bytes_per_pixel": BYTES_PER_PIXEL, "sizes": {}}
    fns = {"y": lambda s, h: hitsir_b200.psnr_ssim_basicsr(s, h, CROP, test_y_channel=True),
           "rgb": lambda s, h: hitsir_b200.psnr_ssim_basicsr(s, h, CROP, test_y_channel=False)}
    for name, ((B, H, W), npairs) in SIZES.items():
        pairs = []
        for _ in range(npairs):
            hr = torch.randint(0, 256, (B, H, W, 3), device=dev, generator=g, dtype=torch.uint8)
            noise = torch.randint(-8, 9, (B, H, W, 3), device=dev, generator=g, dtype=torch.int16)
            pairs.append(((hr.to(torch.int16) + noise).clamp(0, 255).to(torch.uint8), hr))
        by = B * H * W * BYTES_PER_PIXEL
        entry = {"shape": [B, H, W, 3], "rotated_pairs": npairs, "bytes": by}
        for key, f in fns.items():
            ms = time_call(rotating(pairs, f), args.steps, args.warmup, args.window)
            entry[key] = {"ms": round(ms, 4), "gbs": round(by / (ms * 1e-3) / 1e9, 1)}
        res["sizes"][name] = entry
        del pairs
        torch.cuda.empty_cache()

    # tensor2img rounding at cfg2's output: fp32 NCHW read once, uint8 HWC written once (15 bytes per pixel)
    y = torch.rand(32, 3, 1024, 1024, device=dev, generator=g)
    ms = time_call(lambda: hitsir_b200.to_uint8_hwc(y, rounding="nearest"), args.steps, args.warmup, args.window)
    res["round_cfg2"] = {"shape": [32, 3, 1024, 1024], "ms": round(ms, 4), "gbs": round(32 * 1024 * 1024 * 15 / (ms * 1e-3) / 1e9, 1)}
    del y
    torch.cuda.empty_cache()

    torch.manual_seed(0)
    model = hitsir_b200.HiT_SIR(True, True, True, **hitsir_b200.PRO_KWARGS).eval().to(dev)
    x = torch.rand(32, 3, 256, 256, device=dev, generator=g)
    with torch.no_grad():
        t_fwd = time_call(lambda: model(x), 3, 2, args.window)
    res["cfg2_forward_ms"] = round(t_fwd, 2)
    c2 = res["sizes"]["cfg2"]
    res["cfg2_fraction_of_forward"] = {"y": round(c2["y"]["ms"] / t_fwd, 5), "rgb": round(c2["rgb"]["ms"] / t_fwd, 5),
                                       "round": round(res["round_cfg2"]["ms"] / t_fwd, 5)}
    del model, x
    torch.cuda.empty_cache()

    import cv2
    import numpy as np
    from tests import basicsr_ref
    sr, hr = basicsr_ref.inputs("random", 1, 1356, 2040, 1)
    su = basicsr_ref.tensor2img(sr)
    cpu = {}
    for key, yflag in (("y", True), ("rgb", False)):
        t0 = time.perf_counter()
        basicsr_ref.psnr_ssim(su, hr, CROP, yflag)
        cpu[key] = round(time.perf_counter() - t0, 3)
    res["cpu_cv2_div2k_s"] = cpu
    res["cpu"] = {"what": "this host's CPU, cv2/numpy restatement of calculate_psnr + calculate_ssim", "threads": os.cpu_count(),
                  "numpy": np.__version__, "cv2": cv2.__version__}

    info_end = gpu_info(0)
    res["gpu"] = {"name": info["name"], "power_limit_w": info["power_limit_w"], "sm_max_mhz": info["sm_max_mhz"],
                  "sm_mhz_start": info["sm_mhz"], "sm_mhz_end": info_end["sm_mhz"]}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
