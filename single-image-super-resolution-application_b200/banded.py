"""Exact multi-GPU forward of ONE large frame: row bands with halo exchange (SURVEY.md 8f-1).

The reference runs whole frames (test_experiment.py:75, experiments/experiment.py:743); its casa global pools (hit_sir_pro.py:348-349)
and UnionAttention row / column statistics (:124-130) couple every pixel, so the halo-TILED mode of `sharding.ShardedSR.forward_tiled`
is a different function (1.3e-3 away from the full frame even far from the seams, SURVEY.md 0.7).  Here the frame is cut into row
bands whose boundaries are multiples of 192 = lcm(4, 8, 16, 32, 48, 64): no window of any block straddles two bands, so the window
self-correlation is band-local, and what crosses a boundary is exactly
  * 1 row of the bf16 operand of every 3x3 convolution (RHTB convs, conv_after_body, UnionAttention, the upsampler),
  * 2 rows of the FFN hidden map for the depthwise 5x5,
  * 1 row of the per-pixel statistic maps of casa / UnionAttention,
  * an all-reduce of 2 x 180 floats per block (casa pools) and of the UnionAttention column statistics.
The CUDA library asks for these through two callbacks while it enqueues the forward (include/hitsir_b200.h, hitsir_forward_band); this
module provides them in two flavours:

  * `BandedSR`       one band per rank of a torch.distributed group: the workspaces are symmetric memory, a halo exchange is a pair of
                     peer-to-peer copies over NVLink between two device-side barriers, the statistics go through NCCL all-reduces;
  * `LocalBandedSR`  all bands on ONE device, one host thread + one CUDA stream per band, events instead of barriers: the same
                     library path without a second GPU (this is what the single-GPU test suite runs; it is also a way to process a
                     frame whose workspace would not fit in one allocation).
Both return the same frame a single full-frame forward returns, up to the summation order of the all-reduced statistics.
"""
from __future__ import annotations

import ctypes
import threading
from typing import List, Optional, Tuple

import torch

from . import _capi
from .hit_sir_pro import _ws_alloc_bytes, _ws_offset

BAND_UNIT = 192        # lcm of the window sizes 4, 8, 16, 32, 48, 64 (hier_win_ratios x base window 8)
MIN_LAST_BAND = 64     # a band must be longer than its own reflect padding for every window (hit_sir_pro.py:672)


def band_plan(frame_h: int, n_bands: int, unit: int = BAND_UNIT) -> List[Tuple[int, int]]:
    """[(row0, rows)] of at most `n_bands` bands covering [0, frame_h): boundaries are multiples of `unit`, heights differ by at most one
    unit, a short remainder (< MIN_LAST_BAND rows) is merged into the band above it."""
    if frame_h < 1 or n_bands < 1:
        raise ValueError("band_plan needs frame_h >= 1 and n_bands >= 1")
    units = -(-frame_h // unit)
    n = max(1, min(n_bands, units))
    q, r = divmod(units, n)
    bounds = [0]
    for i in range(n):
        bounds.append(bounds[-1] + (q + (1 if i < r else 0)) * unit)
    bounds[-1] = frame_h
    if len(bounds) > 2 and bounds[-1] - bounds[-2] < MIN_LAST_BAND:
        bounds.pop(-2)
    return [(bounds[i], bounds[i + 1] - bounds[i]) for i in range(len(bounds) - 1)]


def _band_struct(frame_h, row0, layout_h, has_top, has_bottom, halo_cb, allreduce_cb):
    b = _capi.HitsirBand()
    b.frame_h, b.row0, b.layout_h, b.has_top, b.has_bottom = frame_h, row0, layout_h, int(has_top), int(has_bottom)
    b.halo, b.allreduce, b.ctx = halo_cb, allreduce_cb, None
    return b


def _forward_band(model, x_frame, y_band, rows, W, band, ws, stream):
    with model._native_call(x_frame.device, ws=ws, stream=stream) as (lib, h, ws_ptr, ws_bytes, st):
        _capi.check(lib.hitsir_forward_band(h, ctypes.c_void_p(x_frame.data_ptr()), ctypes.c_void_p(y_band.data_ptr()), rows, W, ctypes.byref(band),
                                            ws_ptr, ws_bytes, st))


def _workspace_bytes(model, device, layout_h, W) -> int:
    n = ctypes.c_size_t()
    with torch.cuda.device(device):
        _capi.check(_capi.load().hitsir_workspace_bytes_band(model._handle(device), layout_h, W, ctypes.byref(n)))
    return _ws_alloc_bytes(n.value)


class LocalBandedSR:
    """All bands of a frame on one device (see the module docstring).  `n_bands` >= 1."""

    def __init__(self, model, n_bands: int, stat_record: Optional[list] = None, stat_replay: Optional[list] = None):
        """`stat_record`: a list that receives, per all-reduce of the forward, the reduced (sum, max) vectors; `stat_replay`: such a
        list from an earlier run of the same frame, used INSTEAD of this run's reductions (after checking that they agree) -- with it
        a multi-band run and a single-band run see bit-identical statistics, so everything else can be compared bit for bit
        (tests/test_banded.py)."""
        self.model, self.n_bands = model, n_bands
        self.stat_record, self.stat_replay = stat_record, stat_replay
        self.replay_max_rel = 0.0

    def __call__(self, x: torch.Tensor) -> torch.Tensor:
        model = self.model
        if x.dim() != 4 or x.shape[0] != 1 or not x.is_cuda:
            raise RuntimeError("LocalBandedSR expects one CUDA frame (1, C, H, W): there is no CPU path.")
        device = x.device
        x = x.detach().float().contiguous()
        _, C, Hf, W = x.shape
        s = model.out_scale
        plan = band_plan(Hf, self.n_bands)
        R = len(plan)
        layout_h = max(r for _, r in plan)
        cur = torch.cuda.current_stream(device)
        with torch.cuda.device(device):
            h = model._handle(device)
            model._sync_weights(h, device, cur.cuda_stream)
        nbytes = _workspace_bytes(model, device, layout_h, W)
        wss = [torch.empty(nbytes, dtype=torch.uint8, device=device) for _ in range(R)]
        bases = [_ws_offset(w) for w in wss]
        ys = [torch.empty((1, C, s * r, s * W), dtype=torch.float32, device=device) for _, r in plan]
        streams = [torch.cuda.Stream(device) for _ in range(R)]
        for st in streams:
            st.wait_stream(cur)
        rendezvous = threading.Barrier(R)
        ev = [[torch.cuda.Event() for _ in range(2)] for _ in range(R)]
        slots: List[Optional[tuple]] = [None] * R
        calls = [0] * R
        pending_checks: list = []
        errors: List[Optional[BaseException]] = [None] * R

        def view(i, off, nbytes_):
            return wss[i][bases[i] + off: bases[i] + off + nbytes_]

        def make_callbacks(i):
            def neighbours():
                return [j for j in (i - 1, i + 1) if 0 <= j < R]

            def sync_in():          # every band has ENQUEUED everything up to this exchange; make my stream wait for my neighbours' queues
                ev[i][0].record(streams[i])
                rendezvous.wait()
                for j in neighbours():
                    streams[i].wait_event(ev[j][0])

            def sync_out():         # my pushes are enqueued: my neighbours wait for them before they consume their halos
                ev[i][1].record(streams[i])
                rendezvous.wait()
                for j in neighbours():
                    streams[i].wait_event(ev[j][1])
                rendezvous.wait()   # nobody re-records an event a neighbour has not waited on yet

            def halo(_ctx, off, row_bytes, rows, halo_rows, _stream):
                try:
                    with torch.cuda.stream(streams[i]):
                        sync_in()
                        hb = halo_rows * row_bytes
                        if i > 0:       # my first rows -> bottom halo of the band above, which starts right after ITS core rows
                            up_rows = rows * plan[i - 1][1] // plan[i][1]       # buffer rows are proportional to the band heights
                            view(i - 1, off + up_rows * row_bytes, hb).copy_(view(i, off, hb), non_blocking=True)
                        if i < R - 1:   # my last rows -> top halo of the band below
                            view(i + 1, off - hb, hb).copy_(view(i, off + (rows - halo_rows) * row_bytes, hb), non_blocking=True)
                        sync_out()
                    return 0
                except BaseException as e:      # noqa: BLE001 - reported to the C caller as a status, re-raised by __call__
                    errors[i] = e
                    rendezvous.abort()
                    return 1

            def allreduce(_ctx, sum_off, n_sum, max_off, n_max, _stream):
                try:
                    with torch.cuda.stream(streams[i]):
                        sync_in()
                        slots[i] = (view(i, sum_off, 4 * n_sum).view(torch.float32).clone(), view(i, max_off, 4 * n_max).view(torch.float32).clone())
                        ev[i][1].record(streams[i])
                        rendezvous.wait()
                        for j in range(R):
                            streams[i].wait_event(ev[j][1])
                        tot, mx = slots[0]
                        for j in range(1, R):                                              # band order, the same on every band: identical bits
                            tot = tot + slots[j][0]
                            mx = torch.maximum(mx, slots[j][1])
                        k = calls[i]
                        calls[i] += 1
                        if i == 0 and self.stat_record is not None:
                            self.stat_record.append((tot.clone(), mx.clone()))
                        if self.stat_replay is not None:
                            rt, rm = self.stat_replay[k]
                            if i == 0:
                                pending_checks.append((tot, mx, rt, rm))
                            tot, mx = rt, rm
                        view(i, sum_off, 4 * n_sum).view(torch.float32).copy_(tot)
                        view(i, max_off, 4 * n_max).view(torch.float32).copy_(mx)
                        ev[i][0].record(streams[i])
                        rendezvous.wait()
                        for j in range(R):                                                 # slots may be overwritten only after everyone has read them
                            streams[i].wait_event(ev[j][0])
                        rendezvous.wait()
                    return 0
                except BaseException as e:      # noqa: BLE001
                    errors[i] = e
                    rendezvous.abort()
                    return 1
            return _capi.HALO_FN(halo), _capi.ALLREDUCE_FN(allreduce)

        def run(i):
            try:
                row0, rows = plan[i]
                hcb, acb = make_callbacks(i)
                band = _band_struct(Hf, row0, layout_h, i > 0, i < R - 1, hcb, acb)
                with torch.cuda.stream(streams[i]):
                    _forward_band(model, x, ys[i], rows, W, band, wss[i], streams[i].cuda_stream)
            except BaseException as e:          # noqa: BLE001
                if errors[i] is None:
                    errors[i] = e
                rendezvous.abort()

        threads = [threading.Thread(target=run, args=(i,)) for i in range(R)]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        for e in errors:
            if e is not None and not isinstance(e, threading.BrokenBarrierError):
                raise e
        for e in errors:
            if e is not None:
                raise e
        for st in streams:
            cur.wait_stream(st)
        for w in wss + ys:
            w.record_stream(cur)
        for tot, mx, rt, rm in pending_checks:          # how far this run's own reductions are from the replayed ones (summation order only)
            scale = float(rt.abs().max().clamp_min(1e-30))
            self.replay_max_rel = max(self.replay_max_rel, float((tot - rt).abs().max()) / scale,
                                      float((mx - rm).abs().max()) / float(rm.abs().max().clamp_min(1e-30)))
        return torch.cat(ys, dim=2)


class BandedSR:
    """One band per rank of `group` (default: the world).  Construct it collectively on every rank; `forward(x)` takes the SAME whole
    frame on every rank (1, C, H, W) and returns the whole SR frame on `dst_rank` (None elsewhere; every rank when dst_rank is None).
    The group must have exactly len(band_plan(H, world)) ranks (a 1080-row frame has at most 6 bands): build it on a sub-group.

    `graphed=True` captures the band forward of a frame shape -- this rank's ~260 kernel launches TOGETHER with its ~175 exchanges
    (barrier kernels of the symmetric-memory handle, peer copies, NCCL all-reduces) -- into one CUDA graph and replays it: the exchange
    callbacks are Python, and at 6 bands of a 1080p frame a band's kernels last ~100 us each, so the eager path is bound by the host."""

    def __init__(self, model, group=None, graphed: bool = False):
        import torch.distributed as dist
        self.model = model
        self.group = group if group is not None else dist.group.WORLD
        self.world = dist.get_world_size(self.group)
        self.rank = dist.get_rank(self.group)
        self.graphed = graphed
        self._ws = None
        self._key = None
        self._graph = None
        self._gkey = None
        self.captures = 0

    def close(self):
        """Drop the captured graph.  Call it (or delete the object) BEFORE `dist.destroy_process_group()`: tearing down the NCCL
        communicator while a CUDA graph that holds its collectives is alive blocks forever (measured: PyTorch 2.11 / NCCL 2.28)."""
        self._graph = None
        self._gkey = None

    def _workspace(self, device, layout_h, W):
        import torch.distributed._symmetric_memory as symm_mem
        key = (layout_h, W)
        if self._key != key:
            self._graph = None                                                # a captured graph points into the old workspace
            self._gkey = None
            nbytes = _workspace_bytes(self.model, device, layout_h, W)
            self._ws = symm_mem.empty((nbytes,), dtype=torch.uint8, device=device)
            self._hdl = symm_mem.rendezvous(self._ws, self.group)
            self._peers = [self._hdl.get_buffer(p, (nbytes,), torch.uint8) for p in range(self.world)]
            self._key = key
        return self._ws

    def _run_band(self, x, y_band, plan, layout_h):
        """Enqueue this rank's band of the forward (kernels + exchanges) on the current stream."""
        import torch.distributed as dist
        model = self.model
        device = x.device
        _, C, Hf, W = x.shape
        R = len(plan)
        ws = self._ws
        base = _ws_offset(ws)                                                # identical on every rank (symmetric allocations are equally aligned)
        me = self.rank
        hdl, peers = self._hdl, self._peers
        cur = torch.cuda.current_stream(device)

        def halo(_ctx, off, row_bytes, rows, halo_rows, _stream):
            try:
                hb = halo_rows * row_bytes
                hdl.barrier(channel=0)                                       # every band is done with the previous contents of its halos
                if me > 0:
                    up_rows = rows * plan[me - 1][1] // plan[me][1]
                    peers[me - 1][base + off + up_rows * row_bytes: base + off + up_rows * row_bytes + hb].copy_(ws[base + off: base + off + hb], non_blocking=True)
                if me < R - 1:
                    a = base + off + (rows - halo_rows) * row_bytes
                    peers[me + 1][base + off - hb: base + off].copy_(ws[a: a + hb], non_blocking=True)
                hdl.barrier(channel=1)                                       # every push has landed
                return 0
            except BaseException as e:          # noqa: BLE001
                self._err = e
                return 1

        def allreduce(_ctx, sum_off, n_sum, max_off, n_max, _stream):
            try:
                g = self.group
                dist.all_reduce(ws[base + sum_off: base + sum_off + 4 * n_sum].view(torch.float32), op=dist.ReduceOp.SUM, group=g)
                dist.all_reduce(ws[base + max_off: base + max_off + 4 * n_max].view(torch.float32), op=dist.ReduceOp.MAX, group=g)
                return 0
            except BaseException as e:          # noqa: BLE001
                self._err = e
                return 1

        self._err = None
        row0, rows = plan[me]
        hcb, acb = _capi.HALO_FN(halo), _capi.ALLREDUCE_FN(allreduce)
        band = _band_struct(Hf, row0, layout_h, me > 0, me < R - 1, hcb, acb)
        try:
            _forward_band(model, x, y_band, rows, W, band, ws, cur.cuda_stream)
        except Exception:
            if self._err is not None:
                raise self._err
            raise

    def _capture(self, x, plan, layout_h, y_shape):
        device = x.device
        self._graph = None
        self._gx = x.clone()
        self._gy = torch.empty(y_shape, dtype=torch.float32, device=device)
        cur = torch.cuda.current_stream(device)
        side = torch.cuda.Stream(device=device)
        side.wait_stream(cur)
        with torch.cuda.stream(side), torch.no_grad():
            self._run_band(self._gx, self._gy, plan, layout_h)               # eager warm-up: kernels opt in to their shared memory, NCCL connects
            side.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, stream=side, capture_error_mode="thread_local"):
                self._run_band(self._gx, self._gy, plan, layout_h)
        cur.wait_stream(side)
        self._graph = graph
        self.captures += 1

    def forward(self, x: torch.Tensor, dst_rank: Optional[int] = 0) -> Optional[torch.Tensor]:
        import torch.distributed as dist
        model = self.model
        device = x.device
        x = x.detach().float().contiguous()
        _, C, Hf, W = x.shape
        s = model.out_scale
        plan = band_plan(Hf, self.world)
        R = len(plan)
        if R != self.world:          # raised on EVERY rank before anything is enqueued: the exchanges are collective over the group
            raise RuntimeError(f"BandedSR: a frame of {Hf} rows has {R} band(s) of 192-row units but the group has {self.world} ranks; "
                               f"build it on a sub-group of {R} rank(s) (band_plan)")
        layout_h = max(r for _, r in plan)
        cur = torch.cuda.current_stream(device)
        with torch.cuda.device(device):
            h = model._handle(device)
            model._sync_weights(h, device, cur.cuda_stream)
        self._workspace(device, layout_h, W)
        me = self.rank
        y_shape = (1, C, s * plan[me][1], s * W)
        if self.graphed:
            gkey = (tuple(x.shape), model._weights_key(), model.native_handle(device))
            if self._graph is None or self._gkey != gkey:                    # same decision on every rank: same frame, same weights
                self._capture(x, plan, layout_h, y_shape)
                self._gkey = gkey
            self._gx.copy_(x, non_blocking=True)
            self._graph.replay()
            y_band = self._gy
        else:
            y_band = torch.empty(y_shape, dtype=torch.float32, device=device)
            self._run_band(x, y_band, plan, layout_h)
        # reassemble: bands are row blocks of an NCHW tensor
        pad_rows = s * layout_h
        mine = torch.zeros((1, C, pad_rows, s * W), dtype=torch.float32, device=device)
        mine[:, :, : y_band.shape[2]] = y_band
        if dst_rank is None:
            buf = torch.empty((self.world, 1, C, pad_rows, s * W), dtype=torch.float32, device=device)
            dist.all_gather_into_tensor(buf, mine, group=self.group)
        else:
            buf = torch.empty((self.world, 1, C, pad_rows, s * W), dtype=torch.float32, device=device) if me == dst_rank else None
            dist.gather(mine, list(buf.unbind(0)) if me == dst_rank else None, dst=dst_rank, group=self.group)
            if me != dst_rank:
                return None
        return torch.cat([buf[i, :, :, : s * plan[i][1]] for i in range(R)], dim=2)
