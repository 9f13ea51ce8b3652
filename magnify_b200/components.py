"""Reference-facing components: the same names, arguments, exceptions and dataset schema as
magnify's own (`src/magnify/preprocess.py:62-88`, `stitch.py:6-50`, `find.py:13-629`), with the
pixel work done on the GPU through `magnify_b200.ops`.

A component is a callable `Dataset -> Dataset` written against the xarray API: it takes and
returns `xarray.Dataset` when xarray is installed and `magnify_b200.dataset.Dataset` (the same
API, SURVEY.md section 8b "Caveat") when it is not.  `install()` registers the factories in
`magnify.registry.components` under the reference's own names, so `mg.mrbles`, `mg.beads`,
`mg.microfluidic_chip` and their `*_pipe` builders run them unchanged (INTEGRATION.md;
tests/test_dropin_reference.py executes exactly that against the reference's own package).

Hand-off between components stays on the device: what a component stores in the dataset is a
`devarray.DeviceArray` -- the next GPU component takes the tensor from it, the host copy is made
once (pinned memory, copy stream, started in the background) when somebody reads the values.
`flatfield_correct` is lazy like the reference's (there it is a dask graph that executes inside
`stitch`'s cache call, SURVEY.md section 3.1): followed by `stitch` it runs as ONE fused
flat-field + stitch kernel over tiles that are uploaded once, with the maxima pass overlapping
the upload.

Centre finding (`utils.find_circles`, a random search the reference cannot reproduce from run to
run; SURVEY.md section 0 fact 4) runs on the GPU with a seeded sampler (`magnify_b200.circles`,
SURVEY.md section 8f rows N1 / N4); `BeadFinder` / `ButtonFinder` also take a `centers` hook that
pins the centres, which is what the bit-exact ROI / mask parity tests use.
"""
from __future__ import annotations

import math
import os
from dataclasses import dataclass
from typing import Callable, Optional

import numpy as np
import torch

from . import circles, devarray, ops, pipeline
from .devarray import DeviceArray, LazyArray

TILE_DIMS = ("channel", "time", "tile_row", "tile_col", "tile_y", "tile_x")
IMAGE_DIMS = ("channel", "time", "im_y", "im_x")


# ---------------------------------------------------------------------------------------------
# dataset adapters
# ---------------------------------------------------------------------------------------------
def _raw(var):
    """The array object behind a DataArray WITHOUT converting it (NumPy, dask, DeviceArray ...)."""
    return var.data if hasattr(var, "dims") else var


def _to_numpy(var) -> np.ndarray:
    return var.to_numpy() if hasattr(var, "to_numpy") else np.asarray(var)


def _device(device) -> torch.device:
    if not torch.cuda.is_available():
        raise RuntimeError("magnify_b200 components need a CUDA device (there is no CPU fallback)")
    return torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")


def _emit(tensor: torch.Tensor, as_bool: bool = False, extras=None, prefetch: bool = True, name: str = "") -> DeviceArray:
    arr = DeviceArray(tensor, as_bool=as_bool, extras=extras)
    return arr.prefetch() if (prefetch and devarray.PREFETCH and name not in devarray.PREFETCH_SKIP) else arr


def _torch_dtype(np_dtype) -> torch.dtype:
    return torch.from_numpy(np.empty(0, dtype=np.dtype(np_dtype))).dtype


def _is_pinned(arr: np.ndarray) -> bool:
    return arr.size > 0 and arr.flags.c_contiguous and torch.from_numpy(arr.reshape(-1)[:1]).is_pinned()


def _image_on_device(assay, dev) -> torch.Tensor:
    """assay["image"] as a device tensor with 16-byte aligned rows: the tensor `stitch` left there
    (no copy at all), or an upload of host values into an x-padded buffer."""
    data = _raw(assay["image"])
    if isinstance(data, DeviceArray) and data.tensor.device == dev:
        t = data.tensor
        try:
            ops.image_pitch(t)
            return t
        except ValueError:
            out = ops.alloc_image(t.shape, t.dtype, dev)
            out.copy_(t)
            return out
    host = np.ascontiguousarray(_to_numpy(assay["image"]))
    out = ops.alloc_image(host.shape, _torch_dtype(host.dtype), dev)
    src = torch.from_numpy(host)
    out.copy_(src, non_blocking=_is_pinned(host))
    return out


class PendingFlatfield(LazyArray):
    """`flatfield_correct(tile)` not yet evaluated: the raw tile stack plus the flat / dark
    fields.  `stitch` consumes it with the fused kernel; reading it (`np.asarray`) evaluates the
    correction alone on the GPU."""

    def __init__(self, raw, flat, dark, device):
        self.raw, self.flat, self.dark, self.device = raw, flat, dark, device
        self._host = None

    shape = property(lambda self: tuple(self.raw.shape))
    dtype = property(lambda self: np.dtype(self.raw.dtype))

    def numpy(self) -> np.ndarray:
        if self._host is None:
            dev = _device(self.device)
            tiles = _stage_tiles(self.raw, dev, None)
            self._host = ops.flatfield_correct(tiles, self.flat, self.dark).cpu().numpy()
        return self._host


def _stage_tiles(src, dev, ff: Optional[ops.FlatFieldPlan]) -> torch.Tensor:
    """Tile stack (C,T,R,Cc,H,W) -> device tensor, block by (channel, time) block on the copy
    stream, with flat-field pass 1 (`ff`, optional) running on the compute stream as the blocks
    land.  src: DeviceArray (already there), a pinned or pageable NumPy array, a lazily read
    stack with `blocks()` (reader.TiffTiles) or a dask array."""
    maxima = ff is not None and not ff.identity
    if isinstance(src, DeviceArray):
        tiles = src.tensor.contiguous()
        if maxima:
            ops.flatfield_maxima(tiles, ff)
        return tiles
    shape = tuple(int(s) for s in src.shape)
    if len(shape) != 6:
        raise ValueError(f"tile must have 6 dims {TILE_DIMS}, got shape {shape}")
    dtype = _torch_dtype(src.dtype)
    tiles = torch.empty(shape, dtype=dtype, device=dev)
    if tiles.numel() == 0:
        return tiles
    h2d = devarray.Streams.of(dev).h2d
    if isinstance(src, np.ndarray) and _is_pinned(src):
        host = torch.from_numpy(src)
        pipeline.upload_blocks((((ci, ti), host[ci, ti]) for ti in range(shape[1]) for ci in range(shape[0])), tiles,
                               h2d, ff)
    else:
        # pageable memory, dask chunks, TIFF pages: through a ring of pinned slots
        blocks = src.blocks() if callable(getattr(src, "blocks", None)) else pipeline.iter_blocks(src)
        ring = pipeline.PinnedRing(shape[2:], dtype)
        try:
            pipeline.upload_blocks(blocks, tiles, h2d, ff, ring)
        finally:
            ring.close()
    tiles.record_stream(h2d)
    return tiles


def _read_tiff(path) -> np.ndarray:
    """Flat-field / dark-field image file (preprocess.py:75-81 reads it with tifffile): first page,
    through the native TIFF reader."""
    from . import reader

    with reader.TiffFile(os.fspath(path)) as tif:
        return tif.asarray(0)


def _field(value):
    return _read_tiff(os.path.expanduser(value)) if isinstance(value, (str, os.PathLike)) else value


def _check_tile(assay):
    tile = assay["tile"]
    if tuple(tile.dims) != TILE_DIMS:
        raise ValueError(f"tile must have dims {TILE_DIMS} (run standardize_format first), got {tuple(tile.dims)}")
    return tile


# ---------------------------------------------------------------------------------------------
# flatfield_correct  (preprocess.py:62-88)
# ---------------------------------------------------------------------------------------------
def flatfield_correct(xp, flatfield=1.0, darkfield=0.0, device=None):
    tile = _check_tile(xp)
    xp["tile"] = (TILE_DIMS, PendingFlatfield(_raw(tile), _field(flatfield), _field(darkfield), device))
    return xp


def make_flatfield_correct(flatfield=1.0, darkfield=0.0, device=None):
    return lambda xp: flatfield_correct(xp, flatfield=flatfield, darkfield=darkfield, device=device)


# ---------------------------------------------------------------------------------------------
# stitch  (stitch.py:6-50)
# ---------------------------------------------------------------------------------------------
class Stitcher:
    def __init__(self, overlap: int = 102, device=None):
        if overlap < 0:
            raise ValueError("Overlap must be non-negative.")  # stitch.py:8-9
        self.overlap = overlap
        self.device = device
        self._ff = None            # (key, FlatFieldPlan): the device tables of the last flat / dark fields

    def _plan(self, src: "PendingFlatfield", dev) -> ops.FlatFieldPlan:
        key = (id(src.flat), id(src.dark), tuple(src.shape), str(dev))
        if self._ff is None or self._ff[0] != key:
            self._ff = (key, ops.FlatFieldPlan(src.shape, src.flat, src.dark, device=dev), src.flat, src.dark)
        return self._ff[1]

    def __call__(self, assay):
        if "tile" not in assay:
            raise AttributeError("Dataset must contain 'tile' data variable.")  # stitch.py:13-14
        sizes = assay.sizes
        ops.check_overlap(self.overlap, sizes["tile_y"], sizes["tile_x"])  # stitch.py:16-20
        tile = _check_tile(assay)
        dev = _device(self.device)
        src = _raw(tile)
        if isinstance(src, PendingFlatfield) and src._host is None:
            # flatfield_correct + stitch: one upload, the maxima pass under it, one fused kernel
            ff = self._plan(src, dev)
            tiles = _stage_tiles(src.raw, dev, ff)
            image = ops.flatfield_stitch(tiles, overlap=self.overlap, plan=ff, maxima=None if ff.identity else ff.maxima)
        else:
            tiles = _stage_tiles(src.numpy() if isinstance(src, PendingFlatfield) else src, dev, None)
            image = ops.stitch(tiles, self.overlap)
        assay["image"] = (IMAGE_DIMS, _emit(image, name="image"))
        return assay


def make_stitch(overlap: int = 102, device=None):
    return Stitcher(overlap=overlap, device=device)


class FlatfieldStitcher:
    """flatfield_correct + stitch as one component (what the two registered components do when
    they follow each other), for pipelines assembled by hand."""

    def __init__(self, flatfield=1.0, darkfield=0.0, overlap: int = 102, device=None):
        if overlap < 0:
            raise ValueError("Overlap must be non-negative.")
        self.flatfield, self.darkfield = flatfield, darkfield
        self.stitcher = Stitcher(overlap, device)

    def __call__(self, assay):
        if "tile" not in assay:
            raise AttributeError("Dataset must contain 'tile' data variable.")
        raw = assay["tile"]
        out = self.stitcher(flatfield_correct(assay, self.flatfield, self.darkfield, self.stitcher.device))
        out["tile"] = raw          # left as it was (the pipelines drop it, postprocess.py:6-17)
        return out


# ---------------------------------------------------------------------------------------------
# find_beads  (find.py:445-629)
# ---------------------------------------------------------------------------------------------
def _channel_names(assay, n_channels: int):
    return list(_to_numpy(assay["channel"])) if "channel" in assay else list(range(n_channels))


# ---------------------------------------------------------------------------------------------
# marker boxes and masks (find.py:143-181, 380-400, 543-586), shared with pipeline.QuantifyPlan
# ---------------------------------------------------------------------------------------------
# host -> device uploads of the marker code: ops.upload_async, reached through this module so that a
# test can replace it together with `ops`
_upload = ops.upload_async


@dataclass
class Markers:
    """Boxes and masks of M markers over T timepoints, built on the device from host arrays by
    `chip_markers` / `bead_markers` for the finders and for `pipeline.QuantifyPlan`.  Every upload
    is pinned and non-blocking and nothing is read back, so building them never waits behind
    transfers already queued on the device."""
    x: torch.Tensor                    # (M, T) float64 centres
    y: torch.Tensor
    boxes: torch.Tensor                # (M, T, 2) int32 (top, left)
    fg: torch.Tensor                   # (M, Tm, L, L) uint8, one mask per mask timestep
    bg: torch.Tensor
    mask_t: torch.Tensor               # (T,) int32: the mask timestep of every timepoint
    mask_t_host: np.ndarray            # the same as int64 (DeviceArray.take)
    count_bounds: tuple                # upper bounds of the fg / bg pixel counts, from the radii
    labels: Optional[torch.Tensor] = None   # beads: the (Him, Wim) int32 label raster


def _disc_pixels(radius: int) -> int:
    """Pixels of {dx^2 + dy^2 <= r^2}: an upper bound of any disc mask of that radius inside a window."""
    r = int(radius)
    d = np.arange(-r, r + 1)
    return int((d[:, None] ** 2 + d[None, :] ** 2 <= r * r).sum())


def chip_markers(x, y, fg_radius, search_timesteps, chamber_radius: int, max_button_radius: int, roi_length: int,
                 image_shape, device) -> Markers:
    """Chip buttons (find.py:143-181, 380-400): x, y (M, T) float64 centres in image coordinates,
    already copied forward; fg_radius (M, Ts) int, the refined radius or max_button_radius per
    search timestep.  fg is the button disc, bg the annulus max_button_radius < d <= chamber_radius."""
    x = np.asarray(x, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64)
    if x.ndim != 2 or x.shape != y.shape:
        raise ValueError("x and y must have shape (M, T)")
    m, t = x.shape
    src = pipeline.copy_forward_sources(t, search_timesteps)
    search = sorted(set(src.tolist()))
    fg_radius = np.asarray(fg_radius, dtype=np.int32).reshape(m, -1)
    if fg_radius.shape[1] != len(search):
        raise ValueError("fg_radius must have one column per search timestep")
    him, wim = image_shape[-2:]
    xd, yd = _upload(x, device), _upload(y, device)
    boxes, rel = ops.bounding_boxes(xd, yd, roi_length, wim, him, want_rel=True)
    masks = [ops.chip_masks(rel[:, ts].contiguous(), _upload(fg_radius[:, k], device), int(max_button_radius),
                            int(chamber_radius), roi_length) for k, ts in enumerate(search)]
    fg = torch.stack([f for f, _ in masks], 1).contiguous()
    bg = torch.stack([b for _, b in masks], 1).contiguous()
    mask_t = np.searchsorted(search, src).astype(np.int64)                              # find.py:172-173
    bounds = (_disc_pixels(fg_radius.max()) if m else 0,
              max(0, _disc_pixels(chamber_radius) - _disc_pixels(max_button_radius)))
    return Markers(xd, yd, boxes, fg, bg, _upload(mask_t.astype(np.int32), device), mask_t, bounds)


def bead_markers(beads, num_times: int, roi_length: int, image_shape, device) -> Markers:
    """Beads (find.py:543-586): beads (M, 3) rows (row, col, radius), constant over time; fg / bg
    from the label raster, one mask timestep for all timepoints."""
    beads = np.asarray(beads, dtype=np.float64).reshape(-1, 3)
    m, t = len(beads), int(num_times)
    him, wim = image_shape[-2:]
    xd = _upload(np.repeat(beads[:, 1:2], t, axis=1), device)
    yd = _upload(np.repeat(beads[:, 0:1], t, axis=1), device)
    boxes = ops.bounding_boxes(xd, yd, roi_length, wim, him)
    labels = ops.bead_labels(beads.astype(np.int64).astype(np.int32), him, wim, device=device)   # astype(int), find.py:561
    box0 = boxes[:, 0].contiguous() if t > 0 else torch.zeros((m, 2), dtype=torch.int32, device=device)
    fg, bg = ops.bead_masks(labels, box0, roi_length)
    # a bead's fg is at most its own disc (utils.py:398-430), its bg at most the whole window
    rmax = max(int(beads[:, 2].max()), 1) if m else 1
    hw = ops.disc_halfwidth_table(rmax)[rmax]
    bounds = (int((2 * hw + 1).sum() * 2 - (2 * hw[0] + 1)), roi_length * roi_length)
    return Markers(xd, yd, boxes, fg[:, None].contiguous(), bg[:, None].contiguous(),
                   torch.zeros(t, dtype=torch.int32, device=device), np.zeros(t, dtype=np.int64), bounds, labels)


def _gather(image, mk: Markers, length):
    """Crops of every marker, plus the summaries when the image dtype has the fused kernel.  The
    gather's value lists are sized by the markers' count bounds, computed from the radii instead of
    read back from the device: a device->host read here would queue behind the stitched image
    already on its way to the host and stall the whole pipeline for the length of that transfer."""
    if image.dtype == torch.uint16 and mk.boxes.shape[0] > 0:
        return ops.roi_gather_stats(image, mk.boxes, mk.fg, mk.bg, length, mask_t=mk.mask_t, medians=True,
                                    mask_counts=mk.count_bounds)
    return ops.roi_gather(image, mk.boxes, length), None


def _emit_markers(roi_d, stats, mk: Markers):
    """DeviceArrays of the crops and of the (M,T,L,L) masks.  The masks live on the device as their
    distinct timesteps (M,Tm,L,L) and expand lazily; later components find the compact tensors
    and the summaries the gather computed in `extras`."""
    extras = {"stats": stats, "fg": mk.fg, "bg": mk.bg, "mask_t": mk.mask_t}
    roi = _emit(roi_d, extras=extras, name="roi")
    fg = _emit(mk.fg, as_bool=True, extras=extras, prefetch=False).take(mk.mask_t_host, 1)
    bg = _emit(mk.bg, as_bool=True, extras=extras, prefetch=False).take(mk.mask_t_host, 1)
    return roi, fg, bg


class BeadFinder:
    """ROI/mask half of the reference BeadFinder on the GPU (find.py:503-605).

    centers: ndarray (M,3) of (row, col, radius) or a callable `assay -> ndarray` pins the bead
    centres; when omitted they are found on the GPU (`magnify_b200.circles.find_circles`, the
    reference's `utils.find_circles` with a seeded sampler; find.py:476-501)."""

    def __init__(self, min_bead_diameter: int, max_bead_diameter: int, low_edge_quantile: float = 0.1,
                 high_edge_quantile: float = 0.9, num_iter: int = 5000000, min_roundness: float = 0.3,
                 roi_length: Optional[int] = None, search_channel=None, interactive: bool = False,
                 centers=None, device=None, seed: int = 0):
        if min_bead_diameter > max_bead_diameter:
            raise ValueError("min_bead_diameter must be <= max_bead_diameter.")  # find.py:458-459
        self.min_bead_radius = math.floor(min_bead_diameter / 2)
        self.max_bead_radius = math.ceil(max_bead_diameter / 2)
        self.low_edge_quantile, self.high_edge_quantile = low_edge_quantile, high_edge_quantile
        self.num_iter, self.min_roundness = num_iter, min_roundness
        self.roi_length = roi_length if roi_length is not None else 2 * max_bead_diameter  # find.py:467
        self.search_channels = [] if search_channel is None else (
            [search_channel] if isinstance(search_channel, str) else list(search_channel))
        self.interactive = interactive
        self.centers = centers
        self.device = device
        self.seed = seed

    def find_centers(self, assay, image: Optional[torch.Tensor] = None) -> np.ndarray:
        """(M, 3) float64 (row, col, radius): the pinned `centers`, or the GPU circle finder run on
        time 0 of every search channel with the reference's parameters (find.py:476-501)."""
        if self.centers is not None:
            beads = self.centers(assay) if callable(self.centers) else self.centers
            return np.asarray(beads, dtype=np.float64).reshape(-1, 3)
        from scipy.spatial import cKDTree

        dev = _device(self.device)
        if image is None:
            image = _image_on_device(assay, dev)
        names = _channel_names(assay, image.shape[0])
        channels = self.search_channels or names
        beads = np.empty((0, 3))
        for k, ch in enumerate(channels):
            img = circles.to_uint8(image[names.index(ch), 0].contiguous())
            found = circles.find_circles(img, self.low_edge_quantile, self.high_edge_quantile, 20, self.num_iter,
                                         self.min_bead_radius, self.max_bead_radius, self.min_roundness,
                                         self.min_bead_radius, seed=self.seed + k)[0].astype(np.float64)
            if len(beads) > 0 and len(found) > 0:   # drop beads already seen in another channel, find.py:491-500
                near = cKDTree(beads[:, :2]).query_ball_point(found[:, :2], 2 * self.min_bead_radius)
                found = found[~np.array([len(n) > 0 for n in near], dtype=bool)]
            beads = np.concatenate([beads, found])
        return beads

    def __call__(self, assay):
        dev = _device(self.device)
        image = _image_on_device(assay, dev)
        beads = self.find_centers(assay, image)
        c, t = image.shape[:2]
        length = self.roi_length
        m = len(beads)
        x = np.repeat(beads[:, 1:2], t, axis=1)  # find.py:543-550
        y = np.repeat(beads[:, 0:1], t, axis=1)
        valid = np.ones((m, t), dtype=bool)  # find.py:551-554
        if m == 0:  # find.py:557-558
            roi = np.empty((0, c, t, length, length), dtype=np.dtype(assay["image"].dtype))
            fg = np.empty((0, t, length, length), dtype=bool)
            bg = fg.copy()
        else:
            mk = bead_markers(beads, t, length, image.shape, dev)
            roi, fg, bg = _emit_markers(*_gather(image, mk, length), mk)
        assay["roi"] = (("mark", "channel", "time", "roi_y", "roi_x"), roi)
        return assay.assign_coords(
            fg=(("mark", "time", "roi_y", "roi_x"), fg), bg=(("mark", "time", "roi_y", "roi_x"), bg),
            x=(("mark", "time"), x), y=(("mark", "time"), y), valid=(("mark", "time"), valid))


def make_find_beads(min_bead_diameter: int, max_bead_diameter: int, low_edge_quantile: float,
                    high_edge_quantile: float, num_iter: int, min_roundness: float, roi_length: int,
                    search_channel, interactive: bool, centers=None, device=None, seed: int = 0):
    return BeadFinder(min_bead_diameter=min_bead_diameter, max_bead_diameter=max_bead_diameter,
                      low_edge_quantile=low_edge_quantile, high_edge_quantile=high_edge_quantile, num_iter=num_iter,
                      min_roundness=min_roundness, roi_length=roi_length, search_channel=search_channel,
                      interactive=interactive, centers=centers, device=device, seed=seed)


# ---------------------------------------------------------------------------------------------
# find_buttons  (find.py:13-442)
# ---------------------------------------------------------------------------------------------
class ButtonFinder:
    """ROI/mask half of the reference ButtonFinder on the GPU (find.py:143-181, 308-402).

    centers: callable `(assay, t) -> (x, y, fg_radius)` giving, for a search timestep t, the final
    button centres in image coordinates (rows x cols float64 each) and the foreground radii
    (rows x cols int; max_button_radius where refinement found nothing, find.py:363,378).  When
    omitted, centres are found here: full-image circle finding on the GPU, the chip-grid fit on
    the host (`gridfit`), and the per-chamber refinement as one GPU batch
    (find.py:205-306, 336-378; seeded, unlike the reference)."""

    def __init__(self, row_dist: float, col_dist: float, min_button_diameter: int, max_button_diameter: int,
                 chamber_diameter: int, top_chamber=None, left_chamber=None, low_edge_quantile: float = 0.1,
                 high_edge_quantile: float = 0.9, num_iter: int = 5000000, min_roundness: float = 0.20,
                 cluster_penalty: float = 10, roi_length: Optional[int] = None, progress_bar: bool = False,
                 search_timestep=0, search_channel=None, interactive: bool = False, centers: Optional[Callable] = None,
                 device=None, seed: int = 0):
        if min_button_diameter > max_button_diameter:
            raise ValueError("min_button_diameter must be <= max_button_diameter.")  # find.py:34-35
        self.row_dist, self.col_dist = row_dist, col_dist
        self.min_button_radius = math.floor(min_button_diameter / 2)
        self.max_button_radius = math.ceil(max_button_diameter / 2)
        self.chamber_radius = round(chamber_diameter / 2)
        self.roi_length = roi_length if roi_length is not None else round(1.2 * chamber_diameter)  # find.py:49
        self.search_timesteps = sorted(np.atleast_1d(search_timestep).astype(int).tolist())
        self.kwargs = dict(row_dist=row_dist, col_dist=col_dist, min_button_diameter=min_button_diameter,
                           max_button_diameter=max_button_diameter, chamber_diameter=chamber_diameter,
                           top_chamber=top_chamber, left_chamber=left_chamber, low_edge_quantile=low_edge_quantile,
                           high_edge_quantile=high_edge_quantile, num_iter=num_iter, min_roundness=min_roundness,
                           cluster_penalty=cluster_penalty, roi_length=roi_length, progress_bar=progress_bar,
                           search_timestep=search_timestep, search_channel=search_channel, interactive=interactive)
        self.centers = centers
        self.device = device
        self.seed = seed

    def _search_channel_indexes(self, assay, n_channels: int):
        names = _channel_names(assay, n_channels)
        wanted = self.kwargs["search_channel"]
        if wanted is None:
            return list(range(n_channels))
        wanted = [wanted] if isinstance(wanted, str) or np.isscalar(wanted) else list(wanted)
        return [names.index(ch) for ch in wanted]

    def find_centers(self, assay, image: torch.Tensor, t: int):
        """find.py:205-306: circles of every search channel's full image at time t (GPU), merged
        across channels, fitted to the chip grid (host) -> (mark_x, mark_y)."""
        from . import gridfit

        kw = self.kwargs
        tag = _to_numpy(assay["tag"])
        points = np.empty((0, 2))
        for k, ch in enumerate(self._search_channel_indexes(assay, image.shape[0])):
            img = circles.to_uint8(image[ch, t].contiguous())
            found = circles.find_circles(img, kw["low_edge_quantile"], kw["high_edge_quantile"], 20, kw["num_iter"],
                                         self.min_button_radius, self.max_button_radius, kw["min_roundness"],
                                         self.chamber_radius, seed=self.seed + 1000 * t + k)[0]
            points = gridfit.merge_channel_points(points, found[:, :2].astype(np.float64), self.chamber_radius)
        return gridfit.grid_centers(points, tag, tuple(image.shape[-2:]), self.row_dist, self.col_dist,
                                    self.chamber_radius, kw["top_chamber"], kw["left_chamber"], kw["cluster_penalty"])

    def refine(self, assay, image: torch.Tensor, t: int, x: np.ndarray, y: np.ndarray):
        """find.py:324-378: crop every chamber at its grid position, look for the best circle in
        the crop of each search channel (batched on the GPU) and recentre on it.  Returns refined
        x, y (rows, cols) and the foreground radius per chamber (max_button_radius when nothing
        was found or the chamber is blank)."""
        kw = self.kwargs
        dev = image.device
        rows, cols = x.shape
        m, length = rows * cols, self.roi_length
        him, wim = image.shape[-2:]
        tag = _to_numpy(assay["tag"]).reshape(m)
        chans = self._search_channel_indexes(assay, image.shape[0])
        planes = ops.alloc_image((len(chans), 1, him, wim), image.dtype, dev)
        for k, ch in enumerate(chans):
            planes[k, 0].copy_(image[ch, t])
        xd, yd = _upload(x.reshape(m, 1), dev), _upload(y.reshape(m, 1), dev)
        boxes = ops.bounding_boxes(xd, yd, length, wim, him)
        crops = ops.roi_gather(planes, boxes, length)                           # (m, channels, 1, L, L)
        batch = circles.to_uint8(crops.reshape(m * len(chans), length, length), batched=True)   # find.py:343
        high_q = 1 - np.pi * self.min_button_radius / length**2                 # find.py:345-347
        found = circles.find_circles(batch, kw["low_edge_quantile"], high_q, 20, kw["num_iter"] // (rows * cols),
                                     self.min_button_radius, self.max_button_radius, kw["min_roundness"], 0,
                                     seed=self.seed + 1000 * t + 500)
        top_left = boxes[:, 0].cpu().numpy()
        x, y = x.reshape(m).copy(), y.reshape(m).copy()
        radius = np.full(m, self.max_button_radius, dtype=np.int32)
        for i in range(m):
            if tag[i] == "":
                continue
            best, best_score = None, -np.inf
            for k in range(len(chans)):
                cand, scores = found[i * len(chans) + k]
                if len(cand) > 0 and scores[0] > best_score:                    # best first: [0] is the argmax
                    best, best_score = cand[0], scores[0]
            if best is not None:
                y[i], x[i] = best[0] + top_left[i, 0], best[1] + top_left[i, 1]
                radius[i] = best[2]
        return x.reshape(rows, cols), y.reshape(rows, cols), radius

    def _gpu_centers(self, assay, image: torch.Tensor, t: int):
        x, y = self.find_centers(assay, image, t)
        return self.refine(assay, image, t, np.asarray(x, dtype=np.float64), np.asarray(y, dtype=np.float64))

    def __call__(self, assay):
        dev = _device(self.device)
        image = _image_on_device(assay, dev)
        c, t = image.shape[:2]
        rows, cols = assay["tag"].shape
        length = self.roi_length
        find = self.centers if self.centers is not None else (lambda xp, ts: self._gpu_centers(xp, image, ts))
        x, y, radius, src = pipeline.search_centers(lambda ts: find(assay, ts), t, self.search_timesteps)
        mk = chip_markers(x, y, radius, self.search_timesteps, self.chamber_radius, self.max_button_radius, length,
                                   image.shape, dev)
        roi_d, stats = _gather(image, mk, length)
        valid = _to_numpy(assay["valid"]) if "valid" in assay else np.ones((rows, cols, t), dtype=bool)
        valid = valid[:, :, src] if valid.ndim == 3 else valid
        roi, fg, bg = _emit_markers(roi_d, stats, mk)
        x, y = x.reshape(rows, cols, t), y.reshape(rows, cols, t)
        grid = ("mark_row", "mark_col")
        # the reference's layout before its stack (find.py:89-116), then its own stack + transpose (find.py:182)
        assay["roi"] = (grid + ("channel", "time", "roi_y", "roi_x"), roi.reshape(rows, cols, c, t, length, length))
        assay = assay.assign_coords(
            fg=(grid + ("time", "roi_y", "roi_x"), fg.reshape(rows, cols, t, length, length)),
            bg=(grid + ("time", "roi_y", "roi_x"), bg.reshape(rows, cols, t, length, length)),
            x=(grid + ("time",), x), y=(grid + ("time",), y), valid=(grid + ("time",), valid.reshape(rows, cols, t)))
        return assay.stack(mark=grid, create_index=True).transpose("mark", ...)


def make_find_buttons(row_dist, col_dist, min_button_diameter, max_button_diameter, chamber_diameter, top_chamber,
                      left_chamber, low_edge_quantile, high_edge_quantile, num_iter, min_roundness, cluster_penalty,
                      roi_length, progress_bar, search_timestep, search_channel, interactive, centers=None, device=None):
    return ButtonFinder(row_dist, col_dist, min_button_diameter, max_button_diameter, chamber_diameter, top_chamber,
                        left_chamber, low_edge_quantile, high_edge_quantile, num_iter, min_roundness, cluster_penalty,
                        roi_length, progress_bar, search_timestep, search_channel, interactive, centers=centers,
                        device=device)


# ---------------------------------------------------------------------------------------------
# quantify: the per-marker summaries the reference's consumers compute with xarray expressions
# (identify.py:76-80, filter.py:21-22,51,74,82, README.md:21-22)
# ---------------------------------------------------------------------------------------------
def _extras(assay) -> dict:
    data = _raw(assay["roi"])
    return data.extras if isinstance(data, DeviceArray) else {}


def _cached_stats(assay) -> Optional[torch.Tensor]:
    """The summaries the fused gather produced when this package's finder made `roi`."""
    stats = _extras(assay).get("stats")
    if stats is not None and tuple(assay["roi"].dims) == ("mark", "channel", "time", "roi_y", "roi_x") and \
            tuple(stats.shape[:3]) == tuple(assay["roi"].shape[:3]):
        return stats
    return None


def _roi_on_device(assay, dev) -> torch.Tensor:
    """roi for the reductions: uint16 as is; any other dtype the reference accepts (float images,
    tests/test_chip.py:76-96; 8-bit) as float32, which represents uint8 / int16 / float32 exactly."""
    data = _raw(assay["roi"])
    if isinstance(data, DeviceArray) and data.tensor.device == dev:
        t = data.tensor
        if t.dtype not in (torch.uint16, torch.float32):
            t = t.to(torch.float32)
        return t.contiguous()
    host = np.ascontiguousarray(_to_numpy(assay["roi"]))
    if host.dtype not in (np.uint16, np.float32, np.uint8, np.int8, np.int16):
        raise TypeError(f"roi dtype {host.dtype} is not supported by the GPU reductions "
                        "(uint16, float32, 8/16-bit integers)")
    return torch.from_numpy(host if host.dtype in (np.uint16, np.float32) else host.astype(np.float32)).to(dev)


def _masks_on_device(assay, dev):
    """(fg, bg, mask_t): uint8 (M,Tm,L,L) device tensors + the (T,) int32 map of timepoints to them."""
    ex = _extras(assay)
    if all(k in ex and ex[k] is not None for k in ("fg", "bg", "mask_t")) and ex["fg"].device == dev and \
            ex["fg"].shape[0] == assay["roi"].shape[0]:
        return ex["fg"], ex["bg"], ex["mask_t"]
    fg = torch.from_numpy(np.ascontiguousarray(_to_numpy(assay["fg"])).view(np.uint8)).to(dev)
    bg = torch.from_numpy(np.ascontiguousarray(_to_numpy(assay["bg"])).view(np.uint8)).to(dev)
    return fg, bg, torch.arange(fg.shape[1], dtype=torch.int32, device=dev)


def summaries(assay, median: bool = True, device=None) -> torch.Tensor:
    """(M, C, T, 8) float64 summaries (ops.STATS order) of a dataset with roi / fg / bg on the
    stacked `mark` dimension: the ones the gather already produced when `find_buttons` /
    `find_beads` of this package made the roi, else computed from the arrays."""
    dev = _device(device)
    if tuple(assay["roi"].dims) != ("mark", "channel", "time", "roi_y", "roi_x"):
        raise ValueError("quantify needs the stacked schema: roi (mark, channel, time, roi_y, roi_x)")
    cached = _cached_stats(assay)
    if cached is not None:
        return cached
    roi = _roi_on_device(assay, dev)
    if roi.shape[0] == 0:
        return torch.empty(tuple(roi.shape[:3]) + (ops.NSTATS,), dtype=torch.float64, device=dev)
    fg, bg, mask_t = _masks_on_device(assay, dev)
    return ops.roi_stats(roi, fg, bg, mask_t=mask_t, medians=median)


def quantify(assay, median: bool = True, device=None):
    """Adds fg_count/bg_count (mark,time) and fg_sum, bg_sum, fg_mean, bg_mean[, fg_median,
    bg_median] (mark,channel,time): `roi.where(fg).mean(["roi_x","roi_y"])` etc."""
    # the (M,C,T,8) records go to the host once, in the background, BEHIND the crops on the copy stream (a
    # blocking read here would wait for the whole image / roi transfer queued before it on the copy engine and
    # stall the next assay's upload); the variables are lazy column views of that one array
    s = _emit(summaries(assay, median, device), name="summaries")
    dims = ("mark", "channel", "time")
    assay["fg_sum"], assay["bg_sum"] = (dims, s[..., 2]), (dims, s[..., 3])
    assay["fg_mean"], assay["bg_mean"] = (dims, s[..., 4]), (dims, s[..., 5])
    assay["fg_count"], assay["bg_count"] = (("mark", "time"), s[:, 0, :, 0]), (("mark", "time"), s[:, 0, :, 1])
    if median:
        assay["fg_median"], assay["bg_median"] = (dims, s[..., 6]), (dims, s[..., 7])
    return assay


def _time0_medians(assay, channel_index: int, dev):
    """GPU medians of fg and bg at time 0 for one channel -> two (M,) float64 arrays."""
    cached = _cached_stats(assay)
    if cached is not None:
        s = cached[:, channel_index, 0].cpu().numpy()
        return s[:, 6], s[:, 7]
    # copies: host views of pooled / broadcast arrays can be read-only, which torch.from_numpy warns about
    roi = np.array(_to_numpy(assay["roi"])[:, channel_index : channel_index + 1, :1], order="C")
    fg = np.array(_to_numpy(assay["fg"])[:, :1], order="C").view(np.uint8)
    bg = np.array(_to_numpy(assay["bg"])[:, :1], order="C").view(np.uint8)
    roi_d = torch.from_numpy(roi if roi.dtype in (np.uint16, np.float32) else roi.astype(np.float32)).to(dev)
    fgm = ops.roi_median(roi_d, torch.from_numpy(fg).to(dev)).cpu().numpy()[:, 0, 0]
    bgm = ops.roi_median(roi_d, torch.from_numpy(bg).to(dev)).cpu().numpy()[:, 0, 0]
    return fgm, bgm


def _wanted_channels(assay, search_channel):
    channels = _channel_names(assay, assay["roi"].shape[1])
    wanted = channels if search_channel is None else ([search_channel] if isinstance(search_channel, str)
                                                      or np.isscalar(search_channel) else list(search_channel))
    return channels, wanted


def filter_expression(assay, search_channel=None, min_contrast=None, device=None):
    """`filter_expression` of the reference (filter.py:11-37) with the masked medians computed on
    the GPU (SURVEY.md section 8f, row N3).  The pairwise-difference statistic is the reference's
    own expression (O(M^2) on the host, like the reference)."""
    dev = _device(device)
    channels, wanted = _wanted_channels(assay, search_channel)
    valid = _to_numpy(assay["valid"]).astype(bool)
    expressed = np.zeros_like(valid)
    for ch in wanted:
        fgm, bgm = _time0_medians(assay, channels.index(ch), dev)
        if min_contrast is None:
            diffs = bgm[:, np.newaxis] - bgm[np.newaxis, :]
            offdiag = np.ones_like(diffs, dtype=bool) & (~np.eye(len(diffs), dtype=bool))
            upper = 4 * diffs[offdiag].std()
        else:
            upper = min_contrast
        hit = fgm - bgm > upper
        expressed |= hit.reshape((-1,) + (1,) * (valid.ndim - 1))
    return assay.assign_coords(valid=(tuple(assay["valid"].dims), valid & expressed))


def filter_leaky(assay, search_channel=None, device=None):
    """`filter_leaky` of the reference (filter.py:65-94) with the masked medians computed on the
    GPU: tagged markers whose blank neighbour (previous / next mark in stacked order) is not
    "empty" are invalidated.  Needs the stacked chip schema (`tag`, `mark_row` per mark)."""
    dev = _device(device)
    channels, wanted = _wanted_channels(assay, search_channel)
    tag = _to_numpy(assay["tag"])
    rows = _to_numpy(assay["mark_row"])
    valid = _to_numpy(assay["valid"]).astype(bool).copy()
    top = rows.max() if rows.size else 0
    for ch in wanted:
        fgm, bgm = _time0_medians(assay, channels.index(ch), dev)
        diffs = bgm[:, np.newaxis] - bgm[np.newaxis, :]
        offdiag = np.ones_like(diffs, dtype=bool) & (~np.eye(len(diffs), dtype=bool))
        empty = fgm - bgm < 5 * diffs[offdiag].std()
        for i in range(len(tag)):
            if tag[i] == "":
                continue
            if rows[i] > 0 and tag[i - 1] == "":
                valid[i] &= empty[i - 1]
            if rows[i] < top and tag[i + 1] == "":
                valid[i] &= empty[i + 1]
    return assay.assign_coords(valid=(tuple(assay["valid"].dims), valid))


def filter_nonround(assay, min_roundness: float = 0.75, search_channel=None, device=None):
    """`filter_nonround` of the reference (filter.py:40-62): markers whose time-0 foreground has a
    roundness 4 pi area / perimeter^2 not above `min_roundness` (or no contour at all) are
    invalidated.  Perimeters come from the GPU border-following kernel (`ops.mask_perimeters`).  The
    reference repeats the same test once per search channel although `fg` has no channel axis; the
    outcome is that of a single pass."""
    dev = _device(device)
    fg0 = np.array(_to_numpy(assay["fg"])[:, 0], order="C")     # a copy: masks broadcast over time are read-only views
    valid = _to_numpy(assay["valid"]).astype(bool).copy()
    if fg0.shape[0]:
        perimeter = ops.mask_perimeters(torch.from_numpy(fg0.view(np.uint8)).to(dev)).cpu().numpy()
        areas = fg0.sum(axis=(1, 2))
        with np.errstate(divide="ignore", invalid="ignore"):
            roundness = 4 * np.pi * areas.astype(np.float64) / perimeter**2
        keep = (perimeter != 0) & (roundness > min_roundness)
        valid &= keep.reshape((-1,) + (1,) * (valid.ndim - 1))
    return assay.assign_coords(valid=(tuple(assay["valid"].dims), valid))


def mrbles_intensities(assay, channels=None, device=None) -> np.ndarray:
    """The per-bead intensities `identify_mrbles` starts from (identify.py:76-80): mean of the
    foreground minus median of the background at time 0, (mark, channel)."""
    names = _channel_names(assay, assay["roi"].shape[1])
    idx = list(range(len(names))) if channels is None else [names.index(c) for c in channels]
    s = summaries(assay, True, device)[:, :, 0].cpu().numpy()
    return (s[..., 4] - s[..., 7])[:, idx]


def make_quantify(median: bool = True, device=None):
    return lambda xp: quantify(xp, median=median, device=device)


# ---------------------------------------------------------------------------------------------
# registration
# ---------------------------------------------------------------------------------------------
def _component(fn):
    """The reference's `@registry.component` idiom (registry.py:16-29): factory(**kwargs) returns a
    callable that applies `fn(assay, **kwargs)`."""
    return lambda **kwargs: (lambda xp: fn(xp, **kwargs))


FACTORIES = {
    "flatfield_correct": make_flatfield_correct,
    "stitch": make_stitch,
    "find_beads": make_find_beads,
    "find_buttons": make_find_buttons,
    "filter_expression": _component(filter_expression),      # filter.py:11-37
    "filter_nonround": _component(filter_nonround),          # filter.py:40-62
    "filter_leaky": _component(filter_leaky),                # filter.py:65-94
}
EXTRA_FACTORIES = {
    "flatfield_stitch_b200": lambda flatfield=1.0, darkfield=0.0, overlap=102, device=None: FlatfieldStitcher(
        flatfield, darkfield, overlap, device),
    "quantify": make_quantify,
}


def install(override: bool = True, registry=None):
    """Register the GPU components in magnify's component registry (registry.py:12-13).  With
    override the reference's own names are replaced, so the predefined pipelines
    (registry.py:243-269, 431-449, 593-610) use them unchanged; the `<name>_b200` aliases and
    "quantify" are always added.  registry: a catalogue registry (anything with `register(name)`),
    default `magnify.registry.components`."""
    if registry is None:
        try:
            import magnify.registry as mg_registry
        except Exception as e:
            raise ImportError("magnify (and its dependencies xarray, dask, catalogue) must be importable to "
                              "install the magnify_b200 components into its registry") from e
        registry = mg_registry.components
    for name, factory in FACTORIES.items():
        registry.register(name + "_b200")(factory)
        if override:
            registry.register(name)(factory)
    for name, factory in EXTRA_FACTORIES.items():
        registry.register(name)(factory)
    return sorted(list(FACTORIES) + [n + "_b200" for n in FACTORIES] + list(EXTRA_FACTORIES))
