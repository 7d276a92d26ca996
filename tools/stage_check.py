"""Per-stage parity table: CUDA path (tap by tap) vs the CPU oracle.  GPU box only.

    python tools/stage_check.py [--case pro|ablation|ps2|direct3] [--hw 64 64] [--batch 1]
                                [--mode stress|init] [--taps all|coarse]

Prints one line per tap: rel-L2 and max-abs error against the oracle tensor of the same name.
"""
import argparse
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle.weights import synthetic_image  # noqa: E402
from tests.helpers import build_pair, psnr, rel_l2  # noqa: E402

CASES = {
    "pro": ((1, 1, 1), "nearest+conv", 4),
    "ablation": ((0, 0, 0), "nearest+conv", 4),
    "ps2": ((1, 1, 1), "pixelshuffle", 2),
    "ps4": ((1, 0, 1), "pixelshuffle", 4),
    "direct3": ((0, 1, 0), "pixelshuffledirect", 3),
    "direct4": ((1, 1, 0), "pixelshuffledirect", 4),
}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--case", default="pro")
    ap.add_argument("--hw", type=int, nargs=2, default=[64, 64])
    ap.add_argument("--batch", type=int, default=1)
    ap.add_argument("--mode", default="stress")
    ap.add_argument("--taps", default="coarse")
    ap.add_argument("--seed", type=int, default=0)
    args = ap.parse_args()
    flags, up, scale = CASES[args.case]
    model, oracle = build_pair(flags, up, scale, args.mode, args.seed)
    x = synthetic_image(args.batch, args.hw[0], args.hw[1], seed=77)
    taps = {}
    t0 = time.time()
    with torch.no_grad():
        y_ref = oracle.forward(x, taps)
    print(f"oracle forward {time.time() - t0:.1f}s; case={args.case} hw={args.hw} batch={args.batch} mode={args.mode}", flush=True)
    dev = torch.device("cuda:0")
    model = model.to(dev)
    xd = x.to(dev)
    names = list(taps.keys())
    if args.taps == "coarse":
        keep = []
        for n in names:
            if n.startswith("block"):
                i = int(n[5:].split(".")[0])
                if i not in (0,):
                    continue
            keep.append(n)
        names = keep
    worst = 0.0
    for n in names:
        ref = taps[n].contiguous()
        dst = torch.full((ref.numel(),), float("nan"), device=dev)
        model.set_tap(dev, n, dst, stop=True)
        with torch.no_grad():
            model(xd)
        torch.cuda.synchronize()
        got = dst.cpu().view(ref.shape)
        nan = int(torch.isnan(got).sum())
        r = rel_l2(torch.nan_to_num(got), ref)
        m = (torch.nan_to_num(got) - ref).abs().max().item()
        worst = max(worst, r)
        print(f"  {n:28s} shape={tuple(ref.shape)!s:22s} rel_l2={r:.3e} max_abs={m:.3e} ref_absmax={ref.abs().max().item():.3e} nan={nan}", flush=True)
    model.set_tap(dev, None)
    with torch.no_grad():
        y = model(xd)
    torch.cuda.synchronize()
    y = y.cpu()
    print(f"  {'OUTPUT':28s} shape={tuple(y.shape)!s:22s} rel_l2={rel_l2(y, y_ref):.3e} max_abs={(y - y_ref).abs().max().item():.3e} "
          f"psnr={psnr(y, y_ref):.2f}dB nan={int(torch.isnan(y).sum())} launches={model.last_launch_count}", flush=True)
    print(f"worst tap rel_l2 = {worst:.3e}")


if __name__ == "__main__":
    main()
