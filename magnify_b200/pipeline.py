"""Drivers of the hot path over a (channel x time) stack on one GPU (one process per GPU).

`QuantifyPlan` holds everything that is constant over a run (flat/dark tables, marker centres,
boxes, masks) and runs

    tiles --flat-field pass 1 (max)--> [all-reduce MAX] --pass 2 fused with stitch--> image
          --ROI gather fused with masked reductions--> roi, stats

either on tiles already resident in HBM (`QuantifyPlan.run_device`), from pinned host buffers
(`HostStagedRunner.run`: the host->device copies of block k+1 overlap the max pass of block k, and
the device->host copies of one assay overlap the host->device copies of the next), or from an
iterable of pageable chunks such as dask blocks (`ChunkStager.feed` + `HostStagedRunner.finish`).

Time sharding (SURVEY.md section 8e): every rank owns a contiguous block of timepoints; the
only collectives are the all-reduce of the two flat-field maxima and the final gather of the
per-marker summaries (`magnify_b200.dist`).
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Optional

import numpy as np
import torch

from . import ops
from .dist import allreduce_maxima


def copy_forward_sources(num_times: int, search_timesteps) -> np.ndarray:
    """Source timestep of each timestep's centres and masks in ButtonFinder (find.py:143-151):
    the latest search timestep <= t, or the first search timestep for earlier t."""
    search = sorted({int(s) for s in np.atleast_1d(search_timesteps)})
    if not search:
        raise ValueError("at least one search timestep is required")
    if search[0] < 0 or search[-1] >= num_times:
        raise ValueError("search timestep out of range")
    src = np.empty(num_times, dtype=np.int64)
    for t in range(num_times):
        if t < search[0]:
            src[t] = search[0]
        else:
            src[t] = max(s for s in search if s <= t)
    return src


def search_centers(centers_at, num_times: int, search_timesteps):
    """Marker centres at every search timestep, copied forward to the other timepoints
    (find.py:143-157).  centers_at(ts) -> (x, y, fg_radius), M values each in any shape.  Returns
    x, y (M, T) float64, the radii (M, Ts) int32 and the source timestep of every timepoint."""
    src = copy_forward_sources(num_times, search_timesteps)
    search = sorted(set(src.tolist()))
    xs, ys, rs = zip(*(centers_at(ts) for ts in search))
    column = np.searchsorted(search, src)
    x = np.stack([np.asarray(v, dtype=np.float64).reshape(-1) for v in xs], 1)[:, column]
    y = np.stack([np.asarray(v, dtype=np.float64).reshape(-1) for v in ys], 1)[:, column]
    radius = np.stack([np.asarray(v).reshape(-1) for v in rs], 1).astype(np.int32)
    return x, y, radius, src


def upload_blocks(blocks, dst: torch.Tensor, h2d, ff: Optional[ops.FlatFieldPlan] = None, ring=None) -> int:
    """Upload ((channel, time), block) pairs into dst[channel, time] on the copy stream `h2d`; the
    current stream waits for each block and runs flat-field pass 1 (`ff`, skipped when absent or
    the identity) on it as it lands.  A tensor block is copied directly (asynchronously when it is
    pinned); an ndarray or a fill callable goes through the PinnedRing `ring`.  Returns the number
    of blocks."""
    compute = torch.cuda.current_stream(dst.device)
    maxima = ff is not None and not ff.identity
    h2d.wait_stream(compute)          # dst may be overwritten once the kernels queued before are done with it
    if maxima:
        ff.maxima.zero_()
    n = 0
    for (ci, ti), block in blocks:
        if isinstance(block, torch.Tensor):
            with torch.cuda.stream(h2d):
                dst[ci, ti].copy_(block, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(h2d)
        else:
            ev = ring.send(block, dst[ci, ti], h2d)
        compute.wait_event(ev)
        if maxima:
            ops.flatfield_maxima_accumulate(dst[ci, ti], ff, ci)
        n += 1
    return n


@dataclass
class QuantifyResult:
    image: Optional[torch.Tensor]      # (C,T,Him,Wim); dense, or a view padded along x (ops.alloc_image)
    roi: Optional[torch.Tensor]        # (M,C,T,L,L)
    fg: torch.Tensor                   # (M,Tm,L,L) uint8
    bg: torch.Tensor                   # (M,Tm,L,L) uint8
    mask_t: torch.Tensor               # (T,) int32 index into Tm
    boxes: torch.Tensor                # (M,T,2) int32
    stats: torch.Tensor                # (M,C,T,8) float64 in ops.STATS order (medians included)
    maxima: Optional[torch.Tensor] = None
    timings: dict = field(default_factory=dict)


class QuantifyPlan:
    """Static state of one run: tile geometry, flat-field plan, marker boxes and masks."""

    def __init__(self, tile_shape, overlap: int, roi_length: int, flatfield=1.0, darkfield=0.0,
                 device="cuda", group=None):
        self.tile_shape = tuple(int(s) for s in tile_shape)
        c, t, r, cc, h, w = self.tile_shape
        ops.check_overlap(overlap, h, w)
        self.overlap = int(overlap)
        self.roi_length = int(roi_length)
        self.device = torch.device(device)
        self.group = group
        self.image_shape = ops.stitched_shape(self.tile_shape, overlap)
        self.ff = ops.FlatFieldPlan(self.tile_shape, flatfield, darkfield, device=self.device)
        self.boxes = None
        self.order = None
        self.fg = self.bg = self.mask_t = None
        self.mask_counts = None      # (largest fg count, largest bg count): sizes the gather's value lists
        self.medians = True          # per-marker medians are part of the summaries (identify.py:79, filter.py:21-22)

    # -- markers ------------------------------------------------------------------------------
    def set_chip_markers(self, x, y, fg_radius, chamber_radius: int, max_button_radius: int,
                         search_timesteps=0):
        """Chip buttons (ButtonFinder, find.py:55-203 with the centre search done elsewhere).

        x, y: (M, T) float64 centres in image coordinates for every timepoint (non-search
        timepoints hold the copied-forward centres, find.py:156-157,174-175); fg_radius
        (M, Ts) int -- refined radius or max_button_radius per search timestep.  The boxes and
        masks are built as `components.ButtonFinder` builds them (`components.chip_markers`)."""
        from .components import chip_markers

        t = self.tile_shape[1]
        if np.ndim(x) != 2 or np.shape(x)[1] != t or np.shape(x) != np.shape(y):
            raise ValueError(f"x and y must have shape (M, {t})")
        mk = chip_markers(x, y, fg_radius, search_timesteps, chamber_radius, max_button_radius, self.roi_length,
                          self.image_shape, self.device)
        self._set_markers(mk, ops.spatial_order(mk.boxes))
        return self

    def set_bead_markers(self, beads):
        """Beads (BeadFinder, find.py:503-605): beads (M,3) rows (row, col, radius), constant
        over time (find.py:543-550); fg/bg from the label raster (find.py:561-586), built as
        `components.BeadFinder` builds them (`components.bead_markers`)."""
        from .components import bead_markers

        t = self.tile_shape[1]
        mk = bead_markers(beads, t, self.roi_length, self.image_shape, self.device)
        self._set_markers(mk, ops.spatial_order(mk.boxes) if t > 0 else None)
        self.labels = mk.labels
        return self

    def _set_markers(self, mk, order) -> None:
        self.x, self.y, self.boxes, self.fg, self.bg, self.mask_t = mk.x, mk.y, mk.boxes, mk.fg, mk.bg, mk.mask_t
        self.order = order
        # exact counts, read back once: they size the gather's value lists for every run of the plan
        self.mask_counts = ops.mask_count_max(self.fg, self.bg) if mk.boxes.shape[0] else (0, 0)

    def _stage(self, record: Optional[list], name: str, fn):
        """fn(), bracketed by CUDA events on the current stream that are appended to `record` as
        (name, start, end) when a record list is given."""
        if record is None:
            return fn()
        stream = torch.cuda.current_stream(self.device)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        out = fn()
        b.record(stream)
        record.append((name, a, b))
        return out

    # -- markers found on the device-resident image -----------------------------------------------
    def stitched(self, tiles: torch.Tensor, image_out=None, record: Optional[list] = None) -> torch.Tensor:
        """Flat-field + stitch only (the first two stages of run_device): the image the finders
        search, (C, T, Him, Wim) in HBM.  Pass it back to run_device(image=...) to skip the
        recomputation.  record: as in run_device."""
        ff = self.ff
        maxima = None
        if not ff.identity:
            maxima = self._stage(record, "flatfield_max", lambda: ops.flatfield_maxima(tiles, ff))
            if self.group is not None:
                self._stage(record, "allreduce_max", lambda: allreduce_maxima(maxima, self.group))
        return self._stage(record, "flatfield_stitch", lambda: ops.flatfield_stitch(
            tiles, overlap=self.overlap, plan=ff, maxima=maxima, out=image_out))

    def locate_chip_markers(self, image: torch.Tensor, finder, tag, channels=None):
        """Button centres found on the device image by a `components.ButtonFinder` (GPU circle
        finder + host grid fit + batched refinement, find.py:205-378) at its search timesteps,
        copied forward to the others (find.py:143-157), then `set_chip_markers`.  No image bytes
        leave the GPU.  tag: (rows, cols) array of chamber names ("" = blank)."""
        from .dataset import Dataset

        c, t = self.tile_shape[:2]
        tag = np.asarray(tag)
        names = np.asarray(channels if channels is not None else [f"c{k}" for k in range(c)])
        assay = Dataset(coords={"tag": (("mark_row", "mark_col"), tag), "channel": (("channel",), names)})
        x, y, radius, _ = search_centers(lambda ts: finder._gpu_centers(assay, image, ts), t, finder.search_timesteps)
        return self.set_chip_markers(x, y, radius, finder.chamber_radius, finder.max_button_radius,
                                     finder.search_timesteps)

    def locate_bead_markers(self, image: torch.Tensor, finder, channels=None):
        """Bead centres found on the device image by a `components.BeadFinder` (find.py:476-501),
        then `set_bead_markers`."""
        from .dataset import Dataset

        names = np.asarray(channels if channels is not None else [f"c{k}" for k in range(self.tile_shape[0])])
        beads = finder.find_centers(Dataset(coords={"channel": (("channel",), names)}), image)
        return self.set_bead_markers(beads)

    def gather_stats(self, image: torch.Tensor, boxes: torch.Tensor, mask_t: torch.Tensor, **kwargs):
        """`ops.roi_gather_stats` of `image` at `boxes` with the plan's masks, marker order, medians
        and mask counts; kwargs go to it unchanged (want_roi, out_roi, out_stats, peer_stats)."""
        return ops.roi_gather_stats(image, boxes, self.fg, self.bg, self.roi_length, mask_t=mask_t, order=self.order,
                                    medians=self.medians, mask_counts=self.mask_counts, **kwargs)

    # -- device-resident run ------------------------------------------------------------------
    def run_device(self, tiles: torch.Tensor, want_roi: bool = True, image_out=None, roi_out=None,
                   stats_out=None, record: Optional[list] = None, peer_stats=None,
                   image: Optional[torch.Tensor] = None) -> QuantifyResult:
        """Whole hot path on tiles already in HBM (all launches on the current stream).

        record: optional list that receives (stage, start_event, end_event) CUDA-event triples
        recorded on the launching stream (bench.py's per-kernel timing).
        peer_stats: `SymmetricSummaries.peer_blocks` -- the gather kernel then writes the summaries
        into every rank's gathered buffer over NVLink instead of `stats_out` (result.stats is None).
        image: the output of `stitched(tiles)` when it was already computed to locate the markers."""
        if self.boxes is None:
            raise RuntimeError("set_chip_markers / set_bead_markers must be called first")
        if tuple(tiles.shape) != self.tile_shape:
            raise ValueError(f"tiles have shape {tuple(tiles.shape)}, plan was built for {self.tile_shape}")
        maxima = None
        if image is None:
            image = self.stitched(tiles, image_out, record)
            maxima = None if self.ff.identity else self.ff.maxima
        elif tuple(image.shape) != tuple(self.image_shape):
            raise ValueError(f"image has shape {tuple(image.shape)}, plan expects {tuple(self.image_shape)}")
        roi, stats = self._stage(record, "roi_gather_stats", lambda: self.gather_stats(
            image, self.boxes, self.mask_t, want_roi=want_roi, out_roi=roi_out, out_stats=stats_out,
            peer_stats=peer_stats))
        return QuantifyResult(image, roi, self.fg, self.bg, self.mask_t, self.boxes, stats, maxima)


class HostStagedRunner:
    """Pinned-host -> HBM staging loop around a QuantifyPlan (the replacement of the reference's
    dask-chunk reads at find.py:121,155,590 and zarr writes at stitch.py:45, find.py:201,604).

    The host side owns pinned buffers: `tiles_host` (C,T,R,Cc,H,W) in, `image_host`, `roi_host`,
    `stats_host` out.  A copy stream moves the (channel, timepoint) blocks to the GPU while the
    compute stream runs flat-field pass 1 on the blocks that have landed (`upload_blocks`); after
    the maxima all-reduce, pass 2 + gather run on the whole stack and a second copy stream drains
    the results."""

    def __init__(self, plan: QuantifyPlan, want_image: bool = True, want_roi: bool = True):
        self.plan = plan
        c, t, r, cc, h, w = plan.tile_shape
        dev = plan.device
        self.want_image, self.want_roi = want_image, want_roi
        self.tiles_dev = torch.empty(plan.tile_shape, dtype=torch.uint16, device=dev)
        self.image_dev = ops.alloc_image(plan.image_shape, torch.uint16, dev)   # x-padded when Wim % 8 != 0
        m = plan.boxes.shape[0]
        length = plan.roi_length
        self.roi_dev = torch.empty((m, c, t, length, length), dtype=torch.uint16, device=dev) if want_roi else None
        self.stats_dev = torch.empty((m, c, t, ops.NSTATS), dtype=torch.float64, device=dev)
        self.h2d = torch.cuda.Stream(device=dev)
        self.d2h = torch.cuda.Stream(device=dev)
        self.h2d_bytes = self.tiles_dev.numel() * 2
        self.d2h_bytes = self.stats_dev.numel() * 8
        if want_image:
            self.d2h_bytes += self.image_dev.numel() * 2
        if want_roi:
            self.d2h_bytes += self.roi_dev.numel() * 2

    def alloc_host_outputs(self):
        pin = dict(pin_memory=True)
        image = torch.empty(self.plan.image_shape, dtype=torch.uint16, **pin) if self.want_image else None
        roi = torch.empty(tuple(self.roi_dev.shape), dtype=torch.uint16, **pin) if self.want_roi else None
        stats = torch.empty(tuple(self.stats_dev.shape), dtype=torch.float64, **pin)
        return image, roi, stats

    def run(self, tiles_host: torch.Tensor, image_host, roi_host, stats_host) -> None:
        """Enqueue one assay.  Returns as soon as everything is queued: the device->host copies of
        this assay overlap the host->device copies of the next `run()` (PCIe is full duplex), so a
        sequence of assays is bounded by max(H2D, D2H) + compute instead of their sum.  Call
        `synchronize()` before reading the host outputs."""
        c, t = self.plan.tile_shape[:2]
        # stage in + pass 1, time-major: each (channel, time) block is contiguous
        upload_blocks((((ci, ti), tiles_host[ci, ti]) for ti in range(t) for ci in range(c)), self.tiles_dev,
                      self.h2d, self.plan.ff)
        self.finish(image_host, roi_host, stats_host)

    def finish(self, image_host, roi_host, stats_host) -> None:
        """All tiles are on the device and pass 1 has run: all-reduce the maxima, run pass 2 +
        stitch + gather + reductions and queue the device->host copies."""
        plan = self.plan
        ff = plan.ff
        compute = torch.cuda.current_stream(plan.device)
        if not ff.identity and plan.group is not None:
            allreduce_maxima(ff.maxima, plan.group)
        # ---- pass 2 + stitch, gather + reductions on the whole resident stack.  image_dev /
        # roi_dev / stats_dev are reused: wait until the previous assay's results have left them.
        compute.wait_stream(self.d2h)
        image = ops.flatfield_stitch(self.tiles_dev, overlap=plan.overlap, plan=ff,
                                     maxima=None if ff.identity else ff.maxima, out=self.image_dev)
        done_image = torch.cuda.Event()
        done_image.record(compute)
        if self.want_image:
            with torch.cuda.stream(self.d2h):
                self.d2h.wait_event(done_image)
                ops.to_host_dense(image, out=image_host)   # one pitched copy, also for a padded image
        roi, stats = plan.gather_stats(image, plan.boxes, plan.mask_t, want_roi=self.want_roi, out_roi=self.roi_dev,
                                       out_stats=self.stats_dev)
        done_roi = torch.cuda.Event()
        done_roi.record(compute)
        with torch.cuda.stream(self.d2h):
            self.d2h.wait_event(done_roi)
            if self.want_roi:
                roi_host.copy_(roi, non_blocking=True)
            stats_host.copy_(stats, non_blocking=True)

    def synchronize(self) -> None:
        """Wait until every queued assay's results are in the host buffers."""
        self.d2h.synchronize()
        torch.cuda.current_stream(self.plan.device).synchronize()


class PinnedRing:
    """`depth` pinned host slots of one block shape: the hop between memory the copy engine cannot
    read asynchronously (pageable arrays, dask chunks, TIFF pages) and HBM.

    `send(block, dst, stream)` waits until the next slot's previous upload has left it, fills it
    -- `block` is an ndarray (copied by a small thread pool: NumPy copies release the GIL, so the
    pageable->pinned memcpy of block k+1 overlaps the PCIe copy of block k) or a callable
    `fill(slot_array)` that writes the block itself (reader.TiffTiles.blocks: native page reads
    land in the slot, no pageable intermediate) -- and queues the upload into `dst` on `stream`.
    Returns the event recorded after that upload."""

    def __init__(self, block_shape, dtype=torch.uint16, depth: int = 4, threads: int = 4):
        from concurrent.futures import ThreadPoolExecutor

        self.block_shape = tuple(int(s) for s in block_shape)
        self.slots = [torch.empty(self.block_shape, dtype=dtype, pin_memory=True) for _ in range(depth)]
        self.free = [None] * depth
        self.pool = ThreadPoolExecutor(max_workers=threads)
        self.threads = threads
        self.sent = 0

    def _fill(self, slot: int, block) -> None:
        dst = self.slots[slot].numpy()
        if callable(block):
            block(dst)
            return
        src = np.asarray(block)
        if src.shape != dst.shape:
            raise ValueError(f"chunk has shape {src.shape}, expected {dst.shape}")
        if src.dtype != dst.dtype:
            raise TypeError(f"chunk has dtype {src.dtype}, expected {dst.dtype}")
        rows = max(1, dst.shape[0] * (dst.shape[1] if dst.ndim > 1 else 1))
        d2, s2 = dst.reshape((rows, -1)), src.reshape((rows, -1))
        parts = [idx for idx in np.array_split(np.arange(rows), self.threads) if len(idx)]
        list(self.pool.map(lambda idx: np.copyto(d2[idx[0]:idx[-1] + 1], s2[idx[0]:idx[-1] + 1]), parts))

    def send(self, block, dst: torch.Tensor, stream) -> "torch.cuda.Event":
        slot = self.sent % len(self.slots)
        if self.free[slot] is not None:
            self.free[slot].synchronize()
        self._fill(slot, block)
        with torch.cuda.stream(stream):
            dst.copy_(self.slots[slot], non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(stream)
        self.free[slot] = ev
        self.sent += 1
        return ev

    def close(self) -> None:
        for ev in self.free:
            if ev is not None:
                ev.synchronize()
        self.pool.shutdown(wait=True)


class ChunkStager:
    """Chunk provider -> pinned ring -> HBM: the staging loop for tiles that are NOT already in
    pinned memory (the reference's per-page dask chunks, reader.py:265-292, or any iterable of
    NumPy blocks).

    `chunks` yields `((channel, time), block)` with block an ndarray shaped (R, Cc, H, W) -- one
    (channel, timepoint) block of the tile stack, in any order -- or a callable `fill(dst)` that
    writes the block into the pinned slot itself (`reader.TiffTiles.blocks()`).  Flat-field pass 1
    runs on the compute stream as blocks land.  After `feed()` the runner's `finish()` does
    pass 2 + gather + drain."""

    def __init__(self, runner: HostStagedRunner, depth: int = 4, threads: int = 4):
        self.runner = runner
        c, t, r, cc, h, w = runner.plan.tile_shape
        self.ring = PinnedRing((r, cc, h, w), torch.uint16, depth, threads)

    def feed(self, chunks) -> int:
        """Stage every chunk and run flat-field pass 1 on it.  Returns the number of blocks."""
        runner = self.runner
        return upload_blocks(chunks, runner.tiles_dev, runner.h2d, runner.plan.ff, self.ring)

    def close(self):
        self.ring.close()


def iter_blocks(tiles):
    """((channel, time), block) chunks of a (C,T,R,Cc,H,W) array-like (NumPy, or a dask array whose
    chunks are computed block by block) in channel-major order."""
    c, t = tiles.shape[:2]
    for ci in range(c):
        for ti in range(t):
            block = tiles[ci, ti]
            if hasattr(block, "compute"):       # dask: materialise this block only
                block = block.compute()
            yield (ci, ti), block


class StreamingRunner:
    """Two passes over a block source for stacks that fit neither HBM nor host RAM (config 5 as a
    whole is 335 GB): only `depth` timepoints are resident at any time.

    Pass 1 streams every (channel, timepoint) block through a pinned slot into HBM and accumulates
    the two global flat-field maxima (preprocess.py:84,86 need them before any pixel can be
    corrected; skipped for the identity flat-field).  Pass 2 streams the blocks again, one
    timepoint at a time: flat-field + stitch, gather + reductions, and the results of that
    timepoint go back through pinned buffers to `sink`.  The reference does the same two sweeps
    implicitly: its lazy dask graph re-reads every TIFF page for `tiles.max()` and again for the
    corrected tiles (preprocess.py:83-87 on the page-per-chunk array of reader.py:265-292).

    source(c, t, dst): fill the C-contiguous (R, Cc, H, W) array `dst` (a pinned slot) with block
    (c, t) -- e.g. `lambda c, t, dst: tiles.read((c, t), dst)` for a `reader.TiffTiles`.
    sink(t, image, roi, stats): called once per timepoint, in order, with NumPy views of pinned
    buffers that are only valid during the call: image (C, Him, Wim) or None, roi (M, C, L, L) or
    None, stats (M, C, 8)."""

    def __init__(self, plan: QuantifyPlan, depth: int = 2, want_image: bool = True, want_roi: bool = True,
                 threads: int = 4):
        from concurrent.futures import ThreadPoolExecutor

        if plan.boxes is None:
            raise RuntimeError("set_chip_markers / set_bead_markers must be called first")
        self.pool = ThreadPoolExecutor(max_workers=max(1, threads))   # the channels of a timepoint are filled concurrently
        if depth < 2:
            raise ValueError("depth must be at least 2 (one timepoint in flight, one being filled)")
        self.plan, self.depth, self.want_image, self.want_roi = plan, depth, want_image, want_roi
        c, t, r, cc, h, w = plan.tile_shape
        dev = plan.device
        m, length = plan.boxes.shape[0], plan.roi_length
        him, wim = plan.image_shape[-2:]
        pin = dict(pin_memory=True)
        self.tiles_pin = [torch.empty((c, r, cc, h, w), dtype=torch.uint16, **pin) for _ in range(depth)]
        self.tiles_dev = [torch.empty((c, 1, r, cc, h, w), dtype=torch.uint16, device=dev) for _ in range(depth)]
        self.image_dev = [ops.alloc_image((c, 1, him, wim), torch.uint16, dev) for _ in range(depth)]
        self.roi_dev = [torch.empty((m, c, 1, length, length), dtype=torch.uint16, device=dev) if want_roi else None
                        for _ in range(depth)]
        self.stats_dev = [torch.empty((m, c, 1, ops.NSTATS), dtype=torch.float64, device=dev) for _ in range(depth)]
        self.image_pin = [torch.empty((c, 1, him, wim), dtype=torch.uint16, **pin) if want_image else None
                          for _ in range(depth)]
        self.roi_pin = [torch.empty((m, c, 1, length, length), dtype=torch.uint16, **pin) if want_roi else None
                        for _ in range(depth)]
        self.stats_pin = [torch.empty((m, c, 1, ops.NSTATS), dtype=torch.float64, **pin) for _ in range(depth)]
        self.h2d = torch.cuda.Stream(device=dev)
        self.d2h = torch.cuda.Stream(device=dev)
        self.boxes_t = [plan.boxes[:, ti:ti + 1].contiguous() for ti in range(t)]
        self.mask_t = [plan.mask_t[ti:ti + 1].contiguous() if plan.mask_t is not None else None for ti in range(t)]
        self.h2d_bytes = self.d2h_bytes = 0

    def _stage_in(self, source, ti: int, slot: int, consumed) -> "torch.cuda.Event":
        """Fill the slot's pinned tiles from the source and queue their upload."""
        c = self.plan.tile_shape[0]
        if consumed[slot] is not None:
            consumed[slot].synchronize()              # the slot's previous upload has been read by the kernels
        dst = self.tiles_pin[slot].numpy()
        list(self.pool.map(lambda ci: source(ci, ti, dst[ci]), range(c)))   # NumPy copies / native reads drop the GIL
        with torch.cuda.stream(self.h2d):
            self.tiles_dev[slot][:, 0].copy_(self.tiles_pin[slot], non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(self.h2d)
        self.h2d_bytes += self.tiles_pin[slot].numel() * 2
        return ev

    def run(self, source, sink) -> None:
        plan, ff = self.plan, self.plan.ff
        c, t = plan.tile_shape[:2]
        compute = torch.cuda.current_stream(plan.device)
        consumed = [None] * self.depth               # per slot: kernels done reading tiles_dev / tiles_pin uploaded
        self.h2d_bytes = self.d2h_bytes = 0
        # ---- pass 1: global maxima
        if not ff.identity:
            ff.maxima.zero_()
            for ti in range(t):
                slot = ti % self.depth
                up = self._stage_in(source, ti, slot, consumed)
                compute.wait_event(up)
                for ci in range(c):
                    ops.flatfield_maxima_accumulate(self.tiles_dev[slot][ci, 0], ff, ci)
                ev = torch.cuda.Event()
                ev.record(compute)
                consumed[slot] = ev
            if plan.group is not None:
                allreduce_maxima(ff.maxima, plan.group)
        # ---- pass 2: correct + stitch + gather per timepoint, results drained behind the kernels
        drained = [None] * self.depth                # per slot: (timepoint, event after its D2H copies)

        def deliver(slot):
            ti, ev = drained[slot]
            ev.synchronize()
            sink(ti, self.image_pin[slot].numpy()[:, 0] if self.want_image else None,
                 self.roi_pin[slot].numpy()[:, :, 0] if self.want_roi else None, self.stats_pin[slot].numpy()[:, :, 0])
            drained[slot] = None

        for ti in range(t):
            slot = ti % self.depth
            if drained[slot] is not None:
                deliver(slot)                         # frees the slot's device and pinned output buffers
            up = self._stage_in(source, ti, slot, consumed)
            compute.wait_event(up)
            image = ops.flatfield_stitch(self.tiles_dev[slot], overlap=plan.overlap, plan=ff,
                                         maxima=None if ff.identity else ff.maxima, out=self.image_dev[slot])
            roi, stats = plan.gather_stats(image, self.boxes_t[ti], self.mask_t[ti], want_roi=self.want_roi,
                                           out_roi=self.roi_dev[slot], out_stats=self.stats_dev[slot])
            done = torch.cuda.Event()
            done.record(compute)
            consumed[slot] = done
            with torch.cuda.stream(self.d2h):
                self.d2h.wait_event(done)
                if self.want_image:
                    ops.to_host_dense(image, out=self.image_pin[slot])
                    self.d2h_bytes += self.image_pin[slot].numel() * 2
                if self.want_roi:
                    self.roi_pin[slot].copy_(roi, non_blocking=True)
                    self.d2h_bytes += self.roi_pin[slot].numel() * 2
                self.stats_pin[slot].copy_(stats, non_blocking=True)
                self.d2h_bytes += self.stats_pin[slot].numel() * 8
                ev = torch.cuda.Event()
                ev.record(self.d2h)
            drained[slot] = (ti, ev)
        for ti in range(max(0, t - self.depth), t):   # remaining timepoints, in order
            if drained[ti % self.depth] is not None and drained[ti % self.depth][0] == ti:
                deliver(ti % self.depth)
