"""Benchmark of the HiT-SIR-pro forward pass (BASELINE.json metric: output megapixels/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg2|cfg3|cfg4|cfg5|cfg1]
                    [--no-extras] [--no-cpu-baseline] [--gather u8|f32|nccl] [--dump-outputs DIR]

One step = one forward of one batch of synthetic LR images through the public nn.Module (-> C ABI -> CUDA).
N=1 workload: BASELINE.json configs[1] (32 x 3 x 256 x 256 LR, x4 'nearest+conv', pro config).  For N>1 the launcher is torchrun
(one rank per GPU); every rank runs its own batch (weak scaling, no data-path collective) and the SR outputs are gathered to rank 0
over NVLink once per step.  Prints ONE JSON line on rank 0.

Timed region of `value`: K forwards with per-launch profiling OFF, CUDA events on the launching stream, barrier + synchronize on both
sides, max over ranks.  The per-category breakdown / roofline numbers come from a SECOND, profiled pass of a few steps.
Extra keys on the same line (unless --no-extras): "cfg4" = BASELINE configs[3] (16 x 512 x 512, x4) strong-scaled over the N ranks,
"cfg3" = BASELINE configs[2] (the eight 576 x 576 halo tiles of a 1920 x 1080 frame, x2 'pixelshuffle') dealt to the N ranks, gathered
and stitched on rank 0; "gpu_baseline" = the unmodified reference module run eagerly on the same B200 (when HITSIR_REFERENCE_DIR names
a checkout of the original project).
"""
import argparse
import contextlib
import io
import json
import os
import subprocess
import sys
import threading
import time
import warnings

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from oracle.reference import reference_dir  # noqa: E402

WORKLOADS = {
    # name: (flags, upsampler, upscale, batch, H, W, description)
    "cfg1": ((1, 1, 1), "nearest+conv", 4, 1, 64, 64, "HiT-SIR-pro x4, 1x 64x64 LR"),
    "cfg2": ((1, 1, 1), "nearest+conv", 4, 32, 256, 256, "HiT-SIR-pro x4 batched inference, 32x 256x256 LR"),
    "cfg3": ((1, 1, 1), "pixelshuffle", 2, 8, 576, 576, "HiT-SIR-pro x2, the 8 halo tiles (576x576) of a 1920x1080 frame (tile t -> rank t % N)"),
    "cfg4": ((1, 1, 1), "nearest+conv", 4, 16, 512, 512, "hitsir_pro_gan generator x4, 16x 512x512 LR"),
    "cfg5": ((0, 0, 0), "nearest+conv", 4, 32, 256, 256, "ablation HiT-SIR-pro x4 casa=False mulsizeconvextract=False, 32x 256x256 LR"),
}
# algorithmic GFLOP per image of the reference formulation (conv+GEMM+bmm, FMA=2; torch.utils.flop_counter on the
# reference module, SURVEY.md 8d)
GFLOP_PER_IMAGE = {"cfg1": 101.81, "cfg2": 1575.8, "cfg3": 7110.2, "cfg4": 6260.6, "cfg5": 1417.1}
# golden fixture whose "keys" entry lists the reference state_dict (name + shape) of a workload's architecture: lets the reference
# arm build weights without importing the product
KEYS_FIXTURE = {"cfg1": "cfg1_pro_x4_64", "cfg2": "cfg1_pro_x4_64", "cfg4": "cfg1_pro_x4_64", "cfg3": "pro_x2_pixelshuffle_48x36",
                "cfg5": "cfg5_ablation_x4_33x47"}
PRO = dict(embed_dim=180, base_win_size=[8, 8], depths=[6] * 6, num_heads=[6] * 6, mlp_ratio=2, hier_win_ratios=[0.5, 1, 2, 4, 6, 8, 10, 12])


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(bf16=p["bf16_tflops"], bf16_sustained=p.get("bf16_tflops_sustained", p["bf16_tflops"]), hbm=p["hbm_gbs"], src="measured")
    return dict(bf16=1590.0, bf16_sustained=1400.0, hbm=6650.0, src="fallback")


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._halt = threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(float(out[0]))
                self.max_mhz = float(out[1])
                for n, v in zip(names, out[2:]):
                    if v.strip().lower().startswith("active"):
                        self.reasons.add(n)
            except Exception:
                pass
            self._halt.wait(0.1)

    def stop(self):
        self._halt.set()
        self.join(timeout=6)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# analytic algorithmic FLOPs (reference formulation, FMA=2) of one launch of each contraction category
def category_flops(cat, B, H, W):
    N = B * H * W
    table = {
        "gemm_fc1_gelu": 2 * N * 180 * 360, "gemm_fc2_ln": 2 * N * 360 * 180, "gemm_proj_ln": 2 * N * 180 * 180,
        "conv_layer": 2 * N * 9 * 180 * 180, "conv_after_body": 2 * N * 9 * 180 * 180, "conv_ua": 2 * N * 9 * 180 * 180,
        "conv_before_upsample": 2 * N * 9 * 180 * 64, "conv_up1": 2 * 4 * N * 9 * 64 * 64, "conv_up2": 2 * 16 * N * 9 * 64 * 64,
        "conv_hr": 2 * 16 * N * 9 * 64 * 64, "conv_last": 2 * 16 * N * 9 * 64 * 3,
        "conv_hr_last": 2 * 16 * N * 9 * 64 * 64 + 2 * 16 * N * 9 * 64 * 3,
        "gemm_first_msgate": 2 * N * 3 * 180 * (9 + 25 + 49 + 81 + 1), "gemm_first_last": 2 * N * 720 * 180,
        "gemm_first": 2 * N * 27 * 180,
        "ffn_tail": 2 * N * 360 * 180 + 2 * N * 360 * 25,          # fc2 + the depthwise 5x5 (both counted by the reference flop counter)
    }
    if cat in table:
        return table[cat]
    if cat.startswith("scc_w"):
        w = int(cat[5:])
        Hp, Wp = -(-H // w) * w, -(-W // w) * w
        Np = B * Hp * Wp
        Lb = min(w, 8) ** 2
        # k-gen (2 x 15x15 per head), pooling Linear(r^2,1) on k and v, S-SC (q k^T, corr v), C-SC (q^T k, corr v^T)
        return Np * (2 * 2 * 6 * 15 * 15 + 2 * 2 * 90 + 2 * 2 * Lb * 90 + 2 * 2 * 90 * 90)
    return 0


# algorithmic (compulsory, unpadded) HBM bytes of one launch of each bandwidth-bound category: DESIGN.md section 3
def category_bytes(cat, B, H, W):
    N = B * H * W
    table = {
        "ffn_tail": N * (360 * 2 + 180 * 4 + 180 * 4),            # bf16 hidden in, fp32 residual in, fp32 stream out
        "cast_shadow": N * (180 * 4 + 180 * 2),
        "qkv_build": N * (180 * 4 + 180 * 2),                     # fp32 stream in, bf16 window tokens out
        "sca_stats": N * 180 * 4,                                 # fp32 stream in (statistics out are negligible)
        "gemm_proj_ln": N * (180 * 2 + 180 * 4 + 180 * 4 + 180 * 2),   # bf16 A, fp32 residual in, fp32 stream + bf16 shadow out
        "gemm_fc1_gelu": N * (180 * 2 + 360 * 2),
        "ln_rows": N * (180 * 4 + 180 * 4),
        "fusion_combine": N * (5 * 180 * 4 + 180 * 2),
    }
    if cat in table:
        return table[cat]
    if cat.startswith("scc_w"):
        return N * (180 * 2 + 180 * 2)                            # window tokens in (once), self-correlation out
    return 0


def measured_traffic(cat):
    """DRAM bytes per launch of `cat` from the committed ncu capture (profiles/traffic.json), or None."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(path):
        return json.load(open(path)).get(cat)
    return None


def load_reference_class():
    """The reference's own `HiT_SIR` class (models/hit_sir_pro.py:1065), imported unchanged through the 3-symbol timm shim."""
    root = reference_dir()
    if root is None:
        return None
    shim = os.path.join(ROOT, "oracle", "ref_shim")
    for p in (root, shim):
        if p not in sys.path:
            sys.path.insert(0, p)
    warnings.filterwarnings("ignore")
    try:
        with contextlib.redirect_stdout(io.StringIO()):
            from models.hit_sir_pro import HiT_SIR as RefHiT
        return RefHiT
    except Exception as e:                                       # pragma: no cover
        print(f"[bench] reference module not importable from {root}: {type(e).__name__}: {e}", file=sys.stderr)
        return None


def build_reference(RefHiT, flags, up, scale):
    with contextlib.redirect_stdout(io.StringIO()):              # the constructor prints one line per SCC block (:403,405)
        return RefHiT(*[bool(f) for f in flags], upsampler=up, upscale=scale, **PRO).eval()


def gpu_baseline(dev, B=4, H=256, W=256, iters=3):
    """Like-for-like GPU baseline (SURVEY.md 8d): the UNMODIFIED reference module, eager, on the same B200 -- fp32 (PyTorch defaults,
    i.e. TF32 convolutions) and torch.autocast(bf16) -- on a slice of the cfg2 batch.  None when the reference sources are absent."""
    RefHiT = load_reference_class()
    if RefHiT is None:
        return None
    torch.manual_seed(0)
    m = build_reference(RefHiT, (1, 1, 1), "nearest+conv", 4).to(dev)
    x = torch.rand(B, 3, H, W, device=dev)
    out = {"impl": "unmodified reference module (models/hit_sir_pro.py), eager PyTorch on the same GPU", "batch": B, "lr": [H, W]}
    mp = B * 16 * H * W / 1e6

    def timed(ctx):
        with torch.no_grad(), ctx:
            m(x)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(iters):
                m(x)
            e1.record()
            torch.cuda.synchronize()
        return e0.elapsed_time(e1) / iters
    try:
        ms = timed(contextlib.nullcontext())
        out["fp32"] = {"ms": round(ms, 2), "mp_s": round(mp / (ms / 1e3), 2)}
        ms = timed(torch.autocast("cuda", dtype=torch.bfloat16))
        out["autocast_bf16"] = {"ms": round(ms, 2), "mp_s": round(mp / (ms / 1e3), 2)}
    except Exception as e:                                       # pragma: no cover
        out["error"] = f"{type(e).__name__}: {e}"
    del m
    torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------------------------------------------
def timed_steps(step, drain, steps, world, dev, sample_clocks=False):
    """K steps bracketed by barrier + synchronize on both sides, CUDA events on the current (launching) stream; max over ranks."""
    import torch.distributed as dist
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler = ClockSampler(dev.index) if sample_clocks else None
    if sampler:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    drain()                                                     # the last gathers have landed before the clock stops
    e1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    clocks = sampler.stop() if sampler else None
    t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return t.item() / steps, clocks


def make_model(hitsir_b200, workload, dev):
    flags, up, scale, B, H, W, desc = WORKLOADS[workload]
    torch.manual_seed(0)
    kw = dict(hitsir_b200.PRO_KWARGS)
    kw.update(upsampler=up, upscale=scale)
    return hitsir_b200.HiT_SIR(*[bool(f) for f in flags], **kw).eval().to(dev)


def run_cfg4(hitsir_b200, model, dev, world, rank, gather):
    """BASELINE configs[3]: 16 x 512 x 512 LR, x4, STRONG scaling: 16 / N images per rank, uint8 HWC outputs gathered to rank 0."""
    import torch.distributed as dist
    from hitsir_b200.sharding import PeerGather, shard_bounds
    _, _, scale, Bt, H, W, desc = WORKLOADS["cfg4"]
    lo, hi = shard_bounds(Bt, world, rank)
    b = hi - lo
    g = torch.Generator(device=dev)
    g.manual_seed(4321 + rank)
    x = torch.randint(0, 256, (b, H, W, 3), device=dev, dtype=torch.uint8, generator=g)
    peer = PeerGather((b, H * scale, W * scale, 3), torch.uint8, dev, mode="gather", dst=0) if (world > 1 and gather != "nccl" and Bt % world == 0) else None
    buf = torch.empty((Bt, H * scale, W * scale, 3), dtype=torch.uint8, device=dev) if (world > 1 and peer is None and rank == 0) else None
    st = {"i": 0}

    def step():
        y = model.forward_uint8(x)
        if peer is not None:
            peer.start(y, st["i"] & 1)
            st["i"] += 1
        elif world > 1:
            dist.gather(y, list(buf.split(b)) if rank == 0 else None, dst=0)

    def drain():
        if peer is not None:
            peer.wait(0); peer.wait(1)
    with torch.no_grad():
        for _ in range(2):
            step()
        drain()
        ms, _ = timed_steps(step, drain, 3, world, dev)
    mp = Bt * H * scale * W * scale / 1e6
    del peer
    return {"workload": f"cfg4: {desc}; strong scaling, {b} images per GPU; uint8 HWC in/out on the device, outputs gathered to rank 0",
            "ms_per_step": round(ms, 3), "value": round(mp / (ms / 1e3), 3), "unit": "MP/s", "steps": 3, "warmup": 2, "images_per_gpu": b,
            "whole_forward_tflops": round(GFLOP_PER_IMAGE["cfg4"] * Bt / (ms / 1e3) / 1e3, 1)}


def run_cfg3(hitsir_b200, dev, world, rank):
    """BASELINE configs[2]: one 1920 x 1080 frame -> 4K, x2 'pixelshuffle', eight 576 x 576 halo tiles dealt to the ranks
    (KAIR main_test_swinir.py:256-285 tiling), SR tiles gathered over NCCL and stitched on rank 0.  End to end per frame."""
    from hitsir_b200.sharding import ShardedSR, tile_plan
    _, _, scale, _, _, _, desc = WORKLOADS["cfg3"]
    model = make_model(hitsir_b200, "cfg3", dev)
    g = torch.Generator(device=dev)
    g.manual_seed(99)
    frame = torch.rand(1, 3, 1080, 1920, device=dev, generator=g)
    sharded = ShardedSR(model, scale)
    origins = tile_plan(1080, 1920, 576, 72)                   # KAIR stride 504: x origins 0,504,1008,1344; y origins 0,504 -> 8 tiles
    out = {}

    def step():
        out["y"] = sharded.forward_tiled(frame, tile=576, overlap=72, dst_rank=0)
    with torch.no_grad():
        for _ in range(2):
            step()
        ms, _ = timed_steps(step, lambda: None, 3, world, dev)
    if rank == 0:
        assert out["y"].shape == (1, 3, 2160, 3840) and torch.isfinite(out["y"]).all()
    mp = 2160 * 3840 / 1e6
    del model
    torch.cuda.empty_cache()
    return {"workload": f"cfg3: {desc}; {len(origins)} tiles over {world} GPU(s), NCCL gather of the SR tiles + overlap-add stitch on rank 0 inside the timed region",
            "ms_per_frame": round(ms, 3), "value": round(mp / (ms / 1e3), 3), "unit": "MP/s (useful 4K output)", "tiles": len(origins),
            "steps": 3, "warmup": 2, "executed_tflops": round(GFLOP_PER_IMAGE["cfg3"] * len(origins) / (ms / 1e3) / 1e3, 1)}


def run_cfg3_exact(hitsir_b200, dev, world, rank):
    """BASELINE configs[2] as the reference itself runs it -- ONE whole 1920 x 1080 frame (test_experiment.py:75), x2 'pixelshuffle' --
    sharded EXACTLY: row bands on 192-row boundaries, one per rank (at most 6 for 1080 rows), halo rows pushed over NVLink into the
    neighbour's symmetric workspace, casa / UnionAttention statistics all-reduced (hitsir_b200/banded.py).  N = 1: the ordinary forward."""
    import torch.distributed as dist
    from hitsir_b200.banded import BandedSR, band_plan
    model = make_model(hitsir_b200, "cfg3", dev)
    g = torch.Generator(device=dev)
    g.manual_seed(99)
    frame = torch.rand(1, 3, 1080, 1920, device=dev, generator=g)     # the same frame on every rank
    plan = band_plan(1080, world)
    R = len(plan)
    out = {}
    ms_eager = None
    if world > 1:
        grp = dist.new_group(list(range(R)))
        banded = BandedSR(model, group=grp, graphed=False) if rank < R else None

        def step():
            if banded is not None:
                out["y"] = banded.forward(frame, dst_rank=0)
        with torch.no_grad():
            for _ in range(2):
                step()
            ms_eager, _ = timed_steps(step, lambda: None, 3, world, dev)     # exchange callbacks run on the host (Python) every frame
        if banded is not None:
            banded.graphed = True                                            # kernels + exchanges of a band replayed as one CUDA graph
    else:
        def step():
            out["y"] = model(frame)
    with torch.no_grad():
        for _ in range(2):
            step()
        ms, _ = timed_steps(step, lambda: None, 3, world, dev)
    if rank == 0:
        assert out["y"].shape == (1, 3, 2160, 3840) and torch.isfinite(out["y"]).all()
    mp = 2160 * 3840 / 1e6
    if world > 1 and banded is not None:
        banded.close()                       # the captured graph holds NCCL nodes: it must go before the process group does
        del banded
    del model
    torch.cuda.empty_cache()
    return {"workload": f"cfg3 exact: the whole 1920x1080 frame, x2 pixelshuffle, {R} row band(s) {[r for _, r in plan]} over {world} GPU(s); "
                        "halo rows over NVLink peer copies, statistics over NCCL, SR bands gathered to rank 0 inside the timed region",
            "ms_per_frame": round(ms, 3), "value": round(mp / (ms / 1e3), 3), "unit": "MP/s (4K output)", "bands": R, "steps": 3, "warmup": 2,
            "ms_per_frame_eager": None if ms_eager is None else round(ms_eager, 3),
            "note": "ms_per_frame: each band's launches and exchanges replayed as one CUDA graph per rank; ms_per_frame_eager: enqueued per frame (Python exchange callbacks)"}


DUMP_MAX_ELEMENTS = 1 << 23                                     # 32 MiB of float32


def dump_outputs(out_dir, y):
    """Write the SR output `y` of the last timed step as float32 .npy for output-by-output comparison of two builds: `sr.npy` (the
    whole NCHW tensor) when it has at most DUMP_MAX_ELEMENTS values, else `sr_sample.npy`, the values at DUMP_MAX_ELEMENTS flat
    positions drawn (with replacement, sorted) by a generator seeded with 0 -- the same positions for the same output shape."""
    os.makedirs(out_dir, exist_ok=True)
    import numpy as np
    flat = y.detach().reshape(-1)
    if flat.numel() <= DUMP_MAX_ELEMENTS:
        name, arr = "sr", y.detach().float().cpu().numpy()
    else:
        g = torch.Generator().manual_seed(0)
        idx = torch.randint(flat.numel(), (DUMP_MAX_ELEMENTS,), generator=g).sort().values
        name, arr = "sr_sample", flat[idx.to(flat.device)].float().cpu().numpy()
    path = os.path.join(out_dir, name + ".npy")
    np.save(path, arr)
    print(f"[bench] last timed step's output {tuple(y.shape)} -> {path} {arr.shape}", file=sys.stderr)


def run_ours(args):
    import torch.distributed as dist
    import hitsir_b200

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    flags, up, scale, B, H, W, desc = WORKLOADS[args.workload]
    model = make_model(hitsir_b200, args.workload, dev)
    g = torch.Generator(device=dev)
    g.manual_seed(1234 + rank)
    x = torch.rand(B, 3, H, W, device=dev, generator=g)
    out_mp = B * (H * scale) * (W * scale) / 1e6                  # output megapixels per rank per step
    # Output gather (N > 1).  Default "u8": the fp32 result is clipped and converted to uint8 HWC on the device (what the reference's
    # callers do with it, test_experiment.py:75-77) and every rank writes its rows into rank 0's symmetric buffer over NVLink on a side
    # stream, double-buffered, overlapped with the next forward: a GATHER of 1/4 of the fp32 bytes instead of an all-gather.
    # "f32": the same peer-to-peer gather of the fp32 NCHW result; "nccl": one NCCL all_gather_into_tensor of fp32 per step.
    peer, gathered, collective = None, None, "none"
    if world > 1:
        from hitsir_b200.sharding import PeerGather
        mode = args.gather
        try:
            if mode == "u8":
                peer = PeerGather((B, H * scale, W * scale, 3), torch.uint8, dev, mode="gather", dst=0)
                collective = "gather to rank 0 of the uint8 HWC SR outputs: NVLink peer-to-peer copies on a side stream, overlapped with the next forward"
            elif mode == "f32":
                peer = PeerGather((B, 3, H * scale, W * scale), torch.float32, dev, mode="gather", dst=0)
                collective = "gather to rank 0 of the fp32 NCHW SR outputs: NVLink peer-to-peer copies on a side stream"
        except Exception as e:                                  # plumbing fallback only: the compute path is unchanged
            if rank == 0:
                print(f"[bench] PeerGather unavailable ({type(e).__name__}: {e}); using NCCL all_gather", file=sys.stderr)
            peer = None
        ok = torch.tensor([1 if (peer is not None or mode == "nccl") else 0], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)               # all ranks take the same path
        if ok.item() == 0 or mode == "nccl":
            peer, mode = None, "nccl"
            gathered = torch.empty((world * B, 3, H * scale, W * scale), device=dev)
            collective = "NCCL all_gather_into_tensor of the fp32 SR outputs per step"
    state = {"i": 0}
    u8 = world > 1 and peer is not None and args.gather == "u8"

    def step():
        y = model(x)
        if args.dump_outputs:
            state["y"] = y
        if world > 1:
            if peer is not None:
                payload = hitsir_b200.to_uint8_hwc(y) if u8 else y
                peer.start(payload, state["i"] & 1)             # waits (on its own stream) for this forward only
                state["i"] += 1
            else:
                dist.all_gather_into_tensor(gathered, y)
        return y

    def drain():
        if peer is not None:
            peer.wait(0); peer.wait(1)

    with torch.no_grad():
        for _ in range(args.warmup):
            step()
        drain()
        if peer is not None:                                    # untimed check: rank 0 holds what an NCCL gather would deliver
            yv = model(x)
            payload = hitsir_b200.to_uint8_hwc(yv) if u8 else yv
            peer.start(payload, 0)
            got = peer.wait(0)
            ref = [torch.empty_like(payload) for _ in range(world)] if rank == 0 else None
            dist.gather(payload, ref, dst=0)
            if rank == 0 and not torch.equal(got, torch.stack(ref)):
                raise RuntimeError("PeerGather result differs from NCCL gather")
            del ref
        torch.cuda.synchronize()
        launches_per_step = model.last_launch_count
        # ---- the headline: profiling off
        ms_step, clocks = timed_steps(step, drain, args.steps, world, dev, sample_clocks=True)
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, state["y"])
        # ---- second pass, per-launch CUDA events on: per-category breakdown and the dominant kernel's launch time
        psteps = max(1, min(args.steps, 3))
        model.profile_enable(dev, True)
        ms_prof, _ = timed_steps(step, drain, psteps, world, dev)
        prof = model.profile_read(dev)
        model.profile_enable(dev, False)
        # ---- end-to-end through the public host-buffer API: every step copies its inputs from pinned host memory and its result
        # back (HostPipeline: double-buffered, so the PCIe copies of step i overlap the kernels of its neighbours)
        xh = [x.cpu().pin_memory() for _ in range(2)]
        yh = [torch.empty((B, 3, H * scale, W * scale), dtype=torch.float32).pin_memory() for _ in range(2)]
        model.forward_host(xh[0], yh[0])
        pipe = hitsir_b200.HostPipeline(model, dev)
        pipe.submit(xh[0], yh[0])
        pipe.wait()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        n_e2e = max(2, min(args.steps, 6))
        for i in range(n_e2e):
            pipe.submit(xh[i & 1], yh[i & 1])
        pipe.wait()
        e2e_s = (time.perf_counter() - t0) / n_e2e
        del xh, yh, pipe
    t = torch.tensor([e2e_s * 1e3], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms = t[0].item()
    value = world * out_mp / (ms_step / 1e3)
    pk = peaks()
    # dominant kernel category of the step
    cat, (cat_ms, cat_n) = max(prof.items(), key=lambda kv: kv[1][0])
    fl = category_flops(cat, B, H, W)
    by = category_bytes(cat, B, H, W)
    t_launch = cat_ms / cat_n / 1e3
    tflops = fl / t_launch / 1e12 if fl else None
    gbs = by / t_launch / 1e9 if by else None
    # the roofline that binds the dominant kernel: whichever of its two fractions is larger
    f_t = tflops / pk["bf16_sustained"] if tflops else 0.0
    f_h = gbs / pk["hbm"] if gbs else 0.0
    if f_h >= f_t and gbs:
        roof = {"bound": "hbm", "kernel": cat, "achieved": round(gbs, 1), "peak": pk["hbm"], "unit": "GB/s", "frac": round(f_h, 4),
                "algorithmic_bytes_per_launch": by}
    else:
        roof = {"bound": "tensor", "kernel": cat, "achieved": round(tflops, 2) if tflops else None, "peak": pk["bf16_sustained"],
                "unit": "TFLOP/s", "frac": round(f_t, 4) if tflops else None, "algorithmic_flops_per_launch": fl}
    tr = measured_traffic(cat)
    roof["traffic"] = tr.get("bytes_per_launch") if isinstance(tr, dict) else tr
    if isinstance(tr, dict):
        roof["traffic_note"] = tr.get("note")
    whole = GFLOP_PER_IMAGE.get(args.workload, 0) * B / (ms_step / 1e3) / 1e3
    roof.update({"peak_source": pk["src"] + (" (sustained, kernel timed inside a long step)" if roof["bound"] == "tensor" else " (copy bandwidth)"),
                 "kernel_share_of_step": round(cat_ms / (ms_prof * psteps), 3), "launch_ms": round(t_launch * 1e3, 4),
                 "whole_forward_tflops": round(whole, 1), "whole_forward_frac_of_sustained": round(whole / pk["bf16_sustained"], 4),
                 "whole_forward_frac_of_burst": round(whole / pk["bf16"], 4)})
    breakdown = {k: {"ms_per_step": round(v[0] / psteps, 3), "launches_per_step": v[1] // psteps,
                     "tflops": round(category_flops(k, B, H, W) / (v[0] / v[1] / 1e3) / 1e12, 1) if category_flops(k, B, H, W) else None,
                     "gbs": round(category_bytes(k, B, H, W) / (v[0] / v[1] / 1e3) / 1e9, 0) if category_bytes(k, B, H, W) else None}
                 for k, v in sorted(prof.items(), key=lambda kv: -kv[1][0])}
    line = {
        "metric": "HiT-SIR-pro x4 output megapixels/s", "value": round(value, 3), "unit": "MP/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_step, 3), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": f"{args.workload}: {desc}, random-init weights, per-GPU batch {B}",
                   "l2": "activations (>= 0.8 GB per tensor) exceed the 126 MB L2; no explicit flush",
                   "collective": collective,
                   "timing": "headline timed with per-launch profiling off; breakdown / roofline from a second profiled pass of "
                             f"{psteps} step(s) ({round(ms_prof, 3)} ms/step with the event records)"},
        "e2e": {"value": round(world * out_mp / (e2e_ms / 1e3), 3), "unit": "MP/s", "h2d_bytes_per_step": B * 3 * H * W * 4,
                "d2h_bytes_per_step": B * 3 * H * W * scale * scale * 4, "ms_per_step": round(e2e_ms, 3)},
        "gpu_launches": launches_per_step * args.steps,
        "clocks": clocks,
        "roofline": roof,
        "breakdown": breakdown,
    }
    del x
    if not args.no_extras and args.workload == "cfg2":
        model._native.workspaces.clear()
        torch.cuda.empty_cache()
        try:
            line["cfg4"] = run_cfg4(hitsir_b200, model, dev, world, rank, args.gather)
        except Exception as e:                                  # the headline stands even if an extra workload cannot run
            line["cfg4"] = {"error": f"{type(e).__name__}: {e}"}
        model._native.workspaces.clear()
        torch.cuda.empty_cache()
        try:
            line["cfg3"] = run_cfg3(hitsir_b200, dev, world, rank)
        except Exception as e:
            line["cfg3"] = {"error": f"{type(e).__name__}: {e}"}
        torch.cuda.empty_cache()
        try:
            line["cfg3_exact"] = run_cfg3_exact(hitsir_b200, dev, world, rank)
        except Exception as e:
            line["cfg3_exact"] = {"error": f"{type(e).__name__}: {e}"}
    if rank == 0:
        if world == 1 and not args.no_extras:
            model._native.workspaces.clear()
            torch.cuda.empty_cache()
            line["gpu_baseline"] = gpu_baseline(dev)
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(args.workload, budget_s=20.0)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------------------------
def host_threads():
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except (AttributeError, OSError):
        return max(1, os.cpu_count() or 1)


def reference_state_dict(workload, seed=0):
    """Deterministic init-statistics weights with the reference's keys and shapes, from the golden fixture of the architecture."""
    import ast
    import numpy as np
    from oracle.weights import fill_state_dict
    g = np.load(os.path.join(ROOT, "tests", "golden", KEYS_FIXTURE[workload] + ".npz"))
    shapes = {}
    for ln in str(g["keys"]).split("\n"):
        k, shp = ln.split(" ", 1)
        shapes[k] = torch.empty(ast.literal_eval(shp))
    return fill_state_dict(shapes, seed, "init")


def cpu_forward_fn(workload):
    """(callable x -> y on the CPU, kind, description): the UNMODIFIED reference module when its sources are present ("reference"),
    else the oracle port with the relative-position bias rebuilt per forward like the reference does ("port")."""
    flags, up, scale, B, H, W, desc = WORKLOADS[workload]
    RefHiT = load_reference_class()
    if RefHiT is not None:
        torch.manual_seed(0)
        m = build_reference(RefHiT, flags, up, scale)
        return (lambda x: m(x)), "reference", f"unmodified reference module ({reference_dir()}/models/hit_sir_pro.py), fp32, eval, no_grad"
    from oracle.hitsir_oracle import HiTSIROracle, OracleConfig
    o = HiTSIROracle(reference_state_dict(workload), OracleConfig(*[bool(f) for f in flags], upscale=scale, upsampler=up))

    def fwd(x):
        o._bias.clear()                                          # reference semantics: bias tables rebuilt every forward (:477-503)
        return o(x)
    return fwd, "port", ("oracle/hitsir_oracle.py (CPU restatement pinned to the reference's goldens), fp32; the bias rebuild uses separable "
                         "index arithmetic, cheaper than the reference's L^2 x 6 gather, so this port is FASTER than the reference module")


def cpu_baseline(workload, budget_s=20.0):
    """The reference's CPU forward on ONE full-size image of the workload (cfg2: 1 x 3 x 256 x 256 of the 32), all host threads,
    bounded by `budget_s` of timed work (at least 2 forwards after one warm-up)."""
    flags, up, scale, B, H, W, desc = WORKLOADS[workload]
    torch.set_num_threads(host_threads())
    fwd, kind, how = cpu_forward_fn(workload)
    x = torch.rand(1, 3, H, W)
    times = []
    with torch.no_grad():
        fwd(x)
        t_start = time.perf_counter()
        while len(times) < 2 or (time.perf_counter() - t_start < budget_s and len(times) < 5):
            t0 = time.perf_counter()
            fwd(x)
            times.append(time.perf_counter() - t0)
    times.sort()
    med = times[len(times) // 2]
    mp = H * scale * W * scale / 1e6
    return {"value": round(mp / med, 5), "unit": "MP/s", "cores": torch.get_num_threads(), "kind": kind,
            "sample": f"{len(times)} forwards of ONE image 1x3x{H}x{W} LR of the {B}-image {workload} batch (same H x W as the GPU arm), {how}; median {med:.2f} s",
            "seconds_per_forward": round(med, 3)}


def run_reference(args):
    """Reference arm: the reference's own CPU implementation of the path on the box's host cores.  Each step = the forward of ONE
    full-size image of the workload (cfg2: 1 x 3 x 256 x 256), whatever --steps is; the process never imports the product package.
    With the reference sources present (HITSIR_REFERENCE_DIR) the UNMODIFIED module is timed (kind
    "reference"), else the oracle port (kind "port").  Bounded: one warm-up forward, then K timed steps or ~4 minutes, whichever
    comes first (the count actually timed is reported)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    torch.set_num_threads(host_threads())      # torchrun exports OMP_NUM_THREADS=1, which would make the reference arm single-threaded
    flags, up, scale, B, H, W, desc = WORKLOADS[args.workload]
    fwd, kind, how = cpu_forward_fn(args.workload)
    assert "hitsir_b200" not in sys.modules, "the reference arm must not load the product"
    x = torch.rand(1, 3, H, W)
    budget = float(os.environ.get("HITSIR_REF_BUDGET_S", "240"))
    times = []
    with torch.no_grad():
        for _ in range(min(args.warmup, 1)):
            fwd(x)
        t_start = time.perf_counter()
        for _ in range(args.steps):
            t0 = time.perf_counter()
            fwd(x)
            times.append(time.perf_counter() - t0)
            if len(times) >= 2 and time.perf_counter() - t_start > budget:
                break
    dt = sum(times) / len(times)
    mp = H * scale * W * scale / 1e6
    v = round(mp / dt, 5)
    sample = (f"each step = ONE image 1x3x{H}x{W} LR of the {B}x{H}x{W} batch (same config as the GPU arm; 1/{B} of its work per step), "
              f"{how}; {len(times)} of {args.steps} steps timed within the {budget:.0f} s budget, {min(args.warmup, 1)} warm-up")
    print(json.dumps({
        "impl": "reference", "metric": "HiT-SIR-pro x4 output megapixels/s", "value": v, "unit": "MP/s",
        "n_gpus": int(os.environ.get("WORLD_SIZE", "1")), "steps": len(times), "steps_requested": args.steps, "warmup": min(args.warmup, 1),
        "ms_per_step": round(dt * 1e3, 1),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{args.workload}: {desc}, random-init weights, per-GPU batch {B}", "sample": sample},
        "cpu_baseline": {"value": v, "unit": "MP/s", "cores": torch.get_num_threads(), "kind": kind, "sample": sample},
        "e2e": {"value": v, "unit": "MP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=list(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the cfg3 / cfg4 / gpu_baseline keys")
    ap.add_argument("--gather", default=os.environ.get("HITSIR_GATHER", "u8"), choices=["u8", "f32", "nccl"])
    ap.add_argument("--dump-outputs", metavar="DIR", help="write rank 0's SR output of the last timed step to DIR as float32 .npy "
                    "(the whole output up to 32 MiB, else a fixed seeded sample); inputs and weights are seeded, so two builds "
                    "run with the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
