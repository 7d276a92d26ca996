"""Exact multi-GPU sharding of ONE frame by row bands (SURVEY.md 8f-1; hitsir_b200/banded.py, hitsir_forward_band).

CPU part: the partitioning (`band_plan`) and, with world_size 2 over gloo, the exchange protocol the library asks its caller for --
"push my first / last `halo_rows` core rows into the neighbour's halo" + "all-reduce SUM / MAX of a few statistics" -- on a stand-in
network made of the same three ingredient kinds as the real path (a vertical 5-tap stencil, a global mean / max gate, a window-local
operation): banded == whole frame.
GPU part: the real library, all bands on one device (`LocalBandedSR`, one host thread + stream per band) against the ordinary
full-frame forward of the same module -- equal up to the summation order of the all-reduced statistics.
"""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from hitsir_b200.banded import BAND_UNIT, MIN_LAST_BAND, LocalBandedSR, band_plan


@pytest.mark.parametrize("frame_h,n", [(1080, 8), (1080, 4), (1080, 2), (576, 8), (192, 2), (193, 2), (416, 3), (448, 3), (33, 4), (2160, 8)])
def test_band_plan_covers_the_frame_on_window_aligned_boundaries(frame_h, n):
    plan = band_plan(frame_h, n)
    assert 1 <= len(plan) <= n
    assert plan[0][0] == 0 and plan[-1][0] + plan[-1][1] == frame_h
    for (r0, rows), (r1, _) in zip(plan, plan[1:]):
        assert r0 + rows == r1
    for r0, rows in plan[:-1]:
        assert r0 % BAND_UNIT == 0 and rows % BAND_UNIT == 0        # no window of 4 .. 64 straddles a boundary
    assert plan[-1][0] % BAND_UNIT == 0
    if len(plan) > 1:
        assert plan[-1][1] >= MIN_LAST_BAND                          # longer than the reflect padding of every window (:672)
    heights = [r for _, r in plan[:-1]]
    if heights:
        assert max(heights) - min(heights) <= BAND_UNIT


def test_band_plan_examples():
    assert band_plan(1080, 8) == [(0, 192), (192, 192), (384, 192), (576, 192), (768, 192), (960, 120)]
    assert band_plan(1080, 2) == [(0, 576), (576, 504)]
    assert band_plan(416, 3) == [(0, 192), (192, 224)]               # the 32-row remainder joins the band above it
    assert band_plan(100, 4) == [(0, 100)]
    with pytest.raises(ValueError):
        band_plan(0, 2)


# ---- gloo world-2: the exchange protocol on a stand-in network --------------------------------------------------------------------
def _standin_full(x):
    """vertical 5-tap stencil (zero padded) -> gate by global mean / max -> per-192-row-window mean subtraction"""
    H = x.shape[0]
    p = torch.nn.functional.pad(x, (0, 0, 2, 2))
    s = sum((k + 1) * p[k:k + H] for k in range(5))
    g = s * s.mean() + s.amax()
    out = g.clone()
    for r in range(0, H, BAND_UNIT):
        out[r:r + BAND_UNIT] -= g[r:r + BAND_UNIT].mean()
    return out


def _free_port() -> int:
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        Hf, W = 416 + 192, 6
        x = torch.rand(Hf, W, generator=torch.Generator().manual_seed(5), dtype=torch.float64)
        plan = band_plan(Hf, world)
        assert len(plan) == world
        row0, rows = plan[rank]
        layout_h = max(r for _, r in plan)
        halo = 2
        buf = torch.zeros(layout_h + 2 * halo, W, dtype=torch.float64)       # [halo | core (layout_h) | halo], like Bump::take_ext
        buf[halo:halo + rows] = x[row0:row0 + rows]
        # halo exchange (the hitsir_halo_fn contract): first rows -> bottom halo of the band above, last rows -> top halo of the band below
        reqs = []
        if rank > 0:
            reqs.append(dist.isend(buf[halo:2 * halo].clone(), rank - 1))
        if rank < world - 1:
            reqs.append(dist.isend(buf[rows:rows + halo].clone(), rank + 1))
        if rank > 0:
            t = torch.empty(halo, W, dtype=torch.float64); dist.recv(t, rank - 1); buf[0:halo] = t
        if rank < world - 1:
            t = torch.empty(halo, W, dtype=torch.float64); dist.recv(t, rank + 1); buf[halo + rows:2 * halo + rows] = t
        for r in reqs:
            r.wait()
        s = sum((k + 1) * buf[k:k + rows] for k in range(5))
        # all-reduce contract: SUM of the share of the frame mean, MAX of the band maximum
        tot = (s.sum() / (Hf * W)).reshape(1); mx = s.amax().reshape(1)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM); dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        g = s * tot + mx
        out = g.clone()
        for r in range(0, rows, BAND_UNIT):
            out[r:r + BAND_UNIT] -= g[r:r + BAND_UNIT].mean()
        ref = _standin_full(x)[row0:row0 + rows]
        assert torch.allclose(out, ref, rtol=0, atol=1e-12), (out - ref).abs().max()
        open(os.path.join(out_dir, f"ok_{rank}"), "w").close()
    finally:
        dist.destroy_process_group()


def test_world2_gloo_band_exchange_protocol(tmp_path):
    world = 2
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    assert all(os.path.exists(tmp_path / f"ok_{r}") for r in range(world))


# ---- GPU: the library's band mode against its own full-frame forward ----------------------------------------------------------------
# Chain of evidence (floating-point reductions are not associative, and with bf16 operands a 1e-7 change of a pooled statistic flips
# roundings that grow to 1e-4 .. 1e-3 at the output, so "banded == full" cannot be asserted tightly in one step):
#   (1) ordinary forward == the frame run as ONE band, bit for bit (same reduction association);
#   (2) R bands, fed the statistics RECORDED in (1) in place of their own all-reduces == (1), bit for bit: halo rows of every stencil
#       (3x3 convs, depthwise 5x5, casa / UnionAttention statistic maps), window alignment, reflect padding in the last band, frame-level
#       pool multiplicities and the reassembly are exact;
#   (3) the R bands' own all-reduced statistics agree with the recorded ones to summation-order accuracy (1e-5 relative);
#   (4) R bands with their own statistics stay within the bf16 noise of the path (the oracle tolerance) of the ordinary forward.
def _setup(flags, upsampler, upscale, mode, Hf, W, **extra):
    from oracle.weights import synthetic_image
    from tests.helpers import build_pair
    model, oracle = build_pair(flags, upsampler, upscale, mode, 11, **extra)
    return model.to("cuda:0"), oracle, synthetic_image(1, Hf, W, seed=9)


@pytest.mark.gpu
@pytest.mark.parametrize("flags,upsampler,upscale,mode,Hf,W,n_bands,extra", [
    ((1, 1, 1), "nearest+conv", 4, "stress", 416, 72, 3, {}),          # bands 192 + 224 (reflect padding inside the last band)
    ((1, 1, 1), "nearest+conv", 4, "init", 384, 56, 2, {}),            # two full bands, no padding in H
    ((1, 1, 1), "pixelshuffle", 2, "stress", 600, 40, 4, {}),          # 192 x 3 + 24 -> 192, 192, 216
    ((0, 0, 0), "pixelshuffledirect", 3, "stress", 400, 48, 2, {}),    # ablation config: no statistics to all-reduce
    ((1, 1, 1), "nearest+conv", 4, "stress", 420, 64, 2, {"resi_connection": "3conv"}),
    ((0, 1, 1), "nearest+conv", 4, "stress", 400, 48, 2, {"in_chans": 1}),   # MultipleSizeConvExtract needs 3 channels (:59)
])
def test_local_banded_equals_full_frame(flags, upsampler, upscale, mode, Hf, W, n_bands, extra):
    model, _, x = _setup(flags, upsampler, upscale, mode, Hf, W, **extra)
    x = x[:, :extra.get("in_chans", 3)].contiguous().to("cuda:0")
    with torch.no_grad():
        full = model(x)
        rec: list = []
        one = LocalBandedSR(model, 1, stat_record=rec)(x)
        assert torch.equal(one, full)                                                   # (1)
        assert (len(rec) > 0) == bool(flags[1] or flags[2])
        rep = LocalBandedSR(model, n_bands, stat_replay=rec)
        many = rep(x)
        assert many.shape == full.shape and torch.equal(many, full)                     # (2)
        assert rep.replay_max_rel < 1e-5, rep.replay_max_rel                             # (3)
        own = LocalBandedSR(model, n_bands)(x)
    scale = max(1.0, full.abs().max().item())
    err = (own - full).abs().max().item() / scale
    assert err < (6e-2 if mode == "stress" else 3e-3) / 4, err                           # (4)


@pytest.mark.gpu
def test_local_banded_short_frame_is_one_band():
    model, _, x = _setup((1, 1, 1), "nearest+conv", 4, "stress", 100, 64)
    x = x.to("cuda:0")
    with torch.no_grad():
        assert torch.equal(model(x), LocalBandedSR(model, 4)(x))


@pytest.mark.gpu
def test_banded_matches_oracle_where_tiles_do_not():
    """The point of 8f-1: on a frame of two bands the banded forward is as close to the whole-frame oracle as the ordinary forward is,
    while two independent tiles (no statistics / halo exchange) are visibly further away (SURVEY.md 0.7)."""
    from tests.helpers import assert_close
    model, oracle, x = _setup((1, 1, 1), "nearest+conv", 4, "stress", 384, 48)
    with torch.no_grad():
        ref = oracle(x)
        banded = LocalBandedSR(model, 2)(x.to("cuda:0")).cpu()
        tiles = torch.cat([model(x[:, :, :192].to("cuda:0")), model(x[:, :, 192:].to("cuda:0"))], dim=2).cpu()
    assert_close(banded, ref, "stress")
    e_band = (banded - ref).abs().max().item()
    e_tile = (tiles - ref).abs().max().item()
    assert e_tile > 3 * e_band, (e_tile, e_band)


@pytest.mark.gpu
def test_band_mode_rejects_misaligned_bands():
    import ctypes
    from hitsir_b200 import _capi
    from hitsir_b200.banded import _band_struct, _forward_band, _workspace_bytes
    model, _, x = _setup((1, 1, 1), "nearest+conv", 4, "init", 300, 40)
    x = x.to("cuda:0")
    with torch.no_grad():
        model(x[:, :, :64])                       # creates the handle and packs the weights
    ws = torch.empty(_workspace_bytes(model, x.device, 200, 40), dtype=torch.uint8, device=x.device)
    y = torch.empty(1, 3, 800, 160, device=x.device)
    band = _band_struct(300, 100, 200, True, False, _capi.HALO_FN(lambda *a: 0), _capi.ALLREDUCE_FN(lambda *a: 0))
    with pytest.raises(RuntimeError, match="multiples of 192"):
        _forward_band(model, x, y, 200, 40, band, ws, torch.cuda.current_stream().cuda_stream)


# ---- 2 GPUs: one band per rank, symmetric-memory halo pushes over NVLink + NCCL all-reduces (BandedSR) -----------------------------------
def _nccl_worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    import faulthandler
    import sys
    faulthandler.dump_traceback_later(150, exit=True, file=sys.stderr)      # a hung exchange must not hold the GPU box: dump the stacks and exit
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", device_id=dev)
    try:
        from hitsir_b200.banded import BandedSR
        from tests.helpers import build_pair
        from oracle.weights import synthetic_image
        for up, scale, Hf, W in (("nearest+conv", 4, 456, 72), ("pixelshuffle", 2, 384, 40)):
            model, _ = build_pair((1, 1, 1), up, scale, "stress", 11)
            model = model.to(dev)
            x = synthetic_image(1, Hf, W, seed=9).to(dev)
            with torch.no_grad():
                full = model(x)
                y = BandedSR(model).forward(x, dst_rank=None)
                local = LocalBandedSR(model, world)(x)            # the same bands on one device, same library path
            torch.cuda.synchronize()
            assert y.shape == full.shape
            scale_ = max(1.0, full.abs().max().item())
            err_full = (y - full).abs().max().item() / scale_
            err_local = (y - local).abs().max().item() / scale_
            # NCCL's and the local harness's two-operand sums commute, so the two banded runs see identical statistics
            assert err_local == 0.0, err_local
            assert err_full < 6e-2 / 4, err_full
            # the same band forward captured with its exchanges into one CUDA graph and replayed (twice: the barriers hold no state)
            graphed = BandedSR(model, graphed=True)
            with torch.no_grad():
                g1 = graphed.forward(x, dst_rank=None).clone()
                g2 = graphed.forward(x, dst_rank=None)
            torch.cuda.synchronize()
            assert graphed.captures == 1 and torch.equal(g1, y) and torch.equal(g2, y)
            graphed.close()                                   # before destroy_process_group: a live graph with NCCL nodes blocks the teardown
        open(os.path.join(out_dir, f"ok_{rank}"), "w").close()
        faulthandler.cancel_dump_traceback_later()
    finally:
        dist.destroy_process_group()


@pytest.mark.gpu
def test_banded_two_gpus_nvlink(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    world = 2
    mp.spawn(_nccl_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    assert all(os.path.exists(tmp_path / f"ok_{r}") for r in range(world))
