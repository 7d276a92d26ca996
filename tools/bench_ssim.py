"""Timing of the Y-channel SSIM on the device (hitsir_b200.ssim_y), beside psnr_y on the same batches and one cfg2 forward.

    python tools/bench_ssim.py [--steps K] [--warmup W] [--window S]

Prints ONE JSON line with, per size, ms per call of ssim_y with the uniform 7x7 and the Gaussian 11x11 window and of psnr_y; the
achieved GB/s over 24 algorithmic bytes per pixel (two fp32 RGB images read once) and its share of the 7.7 TB/s data-sheet HBM
bandwidth; and at cfg2's output size each metric's time as a fraction of one cfg2 forward (32x3x256x256 LR, x4, pro configuration).
Sizes:
  "div2k":  one DIV2K validation HR image, 1x3x1356x2040.  A pair of such batches is 66 MB and fits in the 126 MB L2, so the calls
            rotate over 4 pairs (264 MB) and read HBM rather than L2;
  "cfg2":   cfg2's output, 32x3x1024x1024 (805 MB per pair, larger than L2 by itself);
  "cfg1":   cfg1's output, 1x3x256x256 (L2-resident and launch-bound: a measure of overheads).
"cpu_oracle_div2k_s" is the float32 numpy/scipy restatement of skimage's structural_similarity (tests/ssim_ref.py) on the DIV2K image,
on this host's CPU, uniform window.
Timed regions: profiling off, CUDA events on the current stream after a synchronize, at least K calls and at least --window seconds
after W warm-up calls.  The GPU name, power limit and SM clocks are read with nvidia-smi in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

HBM_GBS = 7700.0          # HGX B200 data sheet, one GPU (up to 1,000 W)
BYTES_PER_PIXEL = 24      # sr and hr, 3 fp32 channels each
SIZES = {"div2k": ((1, 1356, 2040), 4), "cfg2": ((32, 1024, 1024), 1), "cfg1": ((1, 256, 256), 1)}   # shape, rotated pairs


def gpu_info(index):
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--id={index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                         capture_output=True, text=True, timeout=10).stdout.strip().split(",")
    return dict(zip(["name", "power_limit_w", "sm_mhz", "sm_max_mhz"], [v.strip() for v in out]))


def time_call(fn, steps, warmup, window):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    e1.synchronize()
    one = e0.elapsed_time(e1)
    n = max(steps, min(2000, int(window * 1e3 / max(one, 1e-3)) + 1))
    torch.cuda.synchronize()
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / n


def rotating(pairs, f):
    state = {"i": 0}

    def call():
        sr, hr = pairs[state["i"] % len(pairs)]
        state["i"] += 1
        return f(sr, hr)
    return call


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--window", type=float, default=1.0, help="least seconds per timed region")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_ssim.py needs a CUDA device (B200)")
    import hitsir_b200

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    info = gpu_info(0)
    g = torch.Generator(device=dev)
    g.manual_seed(1234)
    res = {"metric": "ssim_y ms per call", "bytes_per_pixel": BYTES_PER_PIXEL, "hbm_peak_gbs": HBM_GBS, "hbm_peak_src": "HGX B200 data sheet",
           "sizes": {}}
    fns = {"ssim_uniform": lambda s, h: hitsir_b200.ssim_y(s, h),
           "ssim_gaussian": lambda s, h: hitsir_b200.ssim_y(s, h, gaussian_weights=True),
           "psnr": lambda s, h: hitsir_b200.psnr_y(s, h)}
    for name, ((B, H, W), npairs) in SIZES.items():
        pairs = []
        for _ in range(npairs):
            hr = torch.rand(B, 3, H, W, device=dev, generator=g)
            pairs.append((hr + 0.03 * torch.randn(B, 3, H, W, device=dev, generator=g), hr))
        by = B * H * W * BYTES_PER_PIXEL
        entry = {"shape": [B, 3, H, W], "rotated_pairs": npairs, "bytes": by}
        for key, f in fns.items():
            ms = time_call(rotating(pairs, f), args.steps, args.warmup, args.window)
            gbs = by / (ms * 1e-3) / 1e9
            entry[key] = {"ms": round(ms, 4), "gbs": round(gbs, 1), "frac_hbm": round(gbs / HBM_GBS, 3)}
        res["sizes"][name] = entry
        del pairs
        torch.cuda.empty_cache()

    torch.manual_seed(0)
    model = hitsir_b200.HiT_SIR(True, True, True, **hitsir_b200.PRO_KWARGS).eval().to(dev)
    x = torch.rand(32, 3, 256, 256, device=dev, generator=g)
    with torch.no_grad():
        t_fwd = time_call(lambda: model(x), 3, 2, args.window)
    res["cfg2_forward_ms"] = round(t_fwd, 2)
    c2 = res["sizes"]["cfg2"]
    res["cfg2_fraction_of_forward"] = {k: round(c2[k]["ms"] / t_fwd, 5) for k in fns}
    del model, x
    torch.cuda.empty_cache()

    import numpy as np
    from tests import ssim_ref
    sr, hr = ssim_ref.inputs("random", 1, 1356, 2040, 1)
    t0 = time.perf_counter()
    ssim_ref.ssim_y(sr, hr)
    res["cpu_oracle_div2k_s"] = round(time.perf_counter() - t0, 3)
    res["cpu"] = {"what": "this host's CPU, float32 numpy/scipy, uniform window", "threads": os.cpu_count(), "numpy": np.__version__}

    info_end = gpu_info(0)
    res["gpu"] = {"name": info["name"], "power_limit_w": info["power_limit_w"], "sm_max_mhz": info["sm_max_mhz"],
                  "sm_mhz_start": info["sm_mhz"], "sm_mhz_end": info_end["sm_mhz"]}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
