"""Timing of the bicubic resize on the device (hitsir_b200.resize_bicubic), beside a device-to-device copy and one cfg2 forward.

    python tools/bench_resize.py [--steps K] [--warmup W] [--window S]

Prints ONE JSON line with, per case, ms per call, the achieved GB/s over the algorithmic bytes (input read once + output written
once), and its share of the measured copy rate and of the 7.7 TB/s data-sheet HBM bandwidth.  Cases (kernel, input -> output):
  div2k_{pil,matlab}:     one DIV2K validation HR image, 1356x2040 RGB, downscaled by 4 (the LR synthesis of the evaluation);
  cfg2_{pil,matlab}:      cfg2's HR batch, 32x1024x1024 RGB, downscaled by 4 to its LR size 256x256;
  baseline_{pil,matlab}:  the "Bicubic" baseline, cfg2's LR 32x256x256 RGB upscaled by 4 back to 1024x1024.
uint8 HWC for pil, fp32 NCHW for matlab.  Every case rotates over enough inputs that one rotation moves more than the 126 MB L2,
so the timed calls read HBM.  "copy_gbs" is torch's device-to-device copy of 1 GiB (read + write), the attainable streaming rate on
the same card in the same run.  "cfg2_forward_ms" is one forward of the pro configuration on 32x3x256x256 (x4), for scale.
Timed regions: CUDA events on the current stream after a synchronize, at least K calls and at least --window seconds after W
warm-up calls.  The GPU name, power limit and SM clocks are read with nvidia-smi in the same run.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from tools.bench_ssim import gpu_info, time_call  # noqa: E402

HBM_GBS = 7700.0          # HGX B200 data sheet, one GPU (up to 1,000 W)
L2_BYTES = 126 << 20
CASES = {   # name: (kernel, input shape (B, H, W), output size or scale)
    "div2k_pil": ("pil", (1, 1356, 2040), (339, 510)),
    "div2k_matlab": ("matlab", (1, 1356, 2040), 0.25),
    "cfg2_pil": ("pil", (32, 1024, 1024), (256, 256)),
    "cfg2_matlab": ("matlab", (32, 1024, 1024), 0.25),
    "baseline_pil": ("pil", (32, 256, 256), (1024, 1024)),
    "baseline_matlab": ("matlab", (32, 256, 256), 4.0),
}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--window", type=float, default=1.0, help="least seconds per timed region")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_resize.py needs a CUDA device (B200)")
    import hitsir_b200

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    info = gpu_info(0)
    g = torch.Generator(device=dev)
    g.manual_seed(1234)
    res = {"metric": "resize_bicubic ms per call", "hbm_peak_gbs": HBM_GBS, "hbm_peak_src": "HGX B200 data sheet", "cases": {}}

    src = torch.empty(1 << 30, dtype=torch.uint8, device=dev)
    dst = torch.empty_like(src)
    ms = time_call(lambda: dst.copy_(src), args.steps, args.warmup, args.window)
    copy_gbs = 2 * src.numel() / (ms * 1e-3) / 1e9
    res["copy_gbs"] = round(copy_gbs, 1)
    del src, dst

    for name, (kernel, (B, H, W), target) in CASES.items():
        if kernel == "pil":
            make = lambda: torch.randint(0, 256, (B, H, W, 3), dtype=torch.uint8, device=dev, generator=g)   # noqa: E731
            oh, ow = target
            fn = lambda x: hitsir_b200.resize_bicubic(x, size=target, kernel="pil")                          # noqa: E731
            esz = 1
        else:
            make = lambda: torch.rand(B, 3, H, W, device=dev, generator=g)                                    # noqa: E731
            oh, ow = -(-H * target // 1), -(-W * target // 1)
            fn = lambda x: hitsir_b200.resize_bicubic(x, scale=target, kernel="matlab")                      # noqa: E731
            esz = 4
        by = B * 3 * (H * W + int(oh) * int(ow)) * esz
        inputs = [make() for _ in range(max(2, -(-2 * L2_BYTES // by)))]
        state = {"i": 0}

        def call():
            x = inputs[state["i"] % len(inputs)]
            state["i"] += 1
            return fn(x)
        ms = time_call(call, args.steps, args.warmup, args.window)
        gbs = by / (ms * 1e-3) / 1e9
        res["cases"][name] = {"kernel": kernel, "in": [B, H, W, 3], "out": [B, int(oh), int(ow), 3], "rotated_inputs": len(inputs),
                              "bytes": by, "ms": round(ms, 4), "gbs": round(gbs, 1), "frac_copy": round(gbs / copy_gbs, 3),
                              "frac_hbm": round(gbs / HBM_GBS, 3)}
        del inputs
        torch.cuda.empty_cache()

    torch.manual_seed(0)
    model = hitsir_b200.HiT_SIR(True, True, True, **hitsir_b200.PRO_KWARGS).eval().to(dev)
    x = torch.rand(32, 3, 256, 256, device=dev, generator=g)
    with torch.no_grad():
        t_fwd = time_call(lambda: model(x), 3, 2, args.window)
    res["cfg2_forward_ms"] = round(t_fwd, 2)
    res["cfg2_fraction_of_forward"] = {k: round(res["cases"][k]["ms"] / t_fwd, 5) for k in ("cfg2_pil", "cfg2_matlab")}
    del model, x
    torch.cuda.empty_cache()

    info_end = gpu_info(0)
    res["gpu"] = {"name": info["name"], "power_limit_w": info["power_limit_w"], "sm_max_mhz": info["sm_max_mhz"],
                  "sm_mhz_start": info["sm_mhz"], "sm_mhz_end": info_end["sm_mhz"]}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
