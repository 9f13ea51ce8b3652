"""Array-level API of the hot path: torch CUDA tensors in, torch CUDA tensors out.

Every function validates its arguments in Python with the reference's error behaviour, then
launches hand-written sm_100a kernels through the C ABI (include/magnify_b200.h) on torch's
current CUDA stream.  Nothing here computes on the CPU; without a CUDA device or without the
built library the calls raise.

Layouts follow the reference (see SURVEY.md section 8a):
  tiles (C,T,R,Cc,H,W) -> image (C,T,Him,Wim) -> roi (M,C,T,L,L), fg/bg (M,Tm,L,L),
  stats (M,C,T,8) = n_fg, n_bg, sum_fg, sum_bg, mean_fg, mean_bg, median_fg, median_bg.
"""
from __future__ import annotations

import ctypes
from typing import Optional, Sequence

import numpy as np
import torch

from . import _lib

STATS = ("n_fg", "n_bg", "sum_fg", "sum_bg", "mean_fg", "mean_bg", "median_fg", "median_bg")
NSTATS = len(STATS)

_DTYPE_CODE = {
    torch.uint8: _lib.MGB_U8,
    torch.uint16: _lib.MGB_U16,
    torch.float32: _lib.MGB_F32,
    torch.float64: _lib.MGB_F64,
}


_UNSIGNED = (torch.uint8, torch.uint16)


def _stream() -> ctypes.c_void_p:
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t: Optional[torch.Tensor]) -> ctypes.c_void_p:
    return ctypes.c_void_p(0 if t is None else t.data_ptr())


def _check(t: torch.Tensor, name: str, dtype=None, ndim=None) -> torch.Tensor:
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor, got {type(t).__name__}")
    if not t.is_cuda:
        raise RuntimeError(f"{name} must live on a CUDA device (magnify_b200 has no CPU path)")
    if dtype is not None and t.dtype != dtype:
        raise TypeError(f"{name} must have dtype {dtype}, got {t.dtype}")
    if ndim is not None and t.dim() != ndim:
        raise ValueError(f"{name} must have {ndim} dimensions, got shape {tuple(t.shape)}")
    if not t.is_contiguous():
        raise ValueError(f"{name} must be contiguous")
    return t


def sm_count() -> int:
    return _lib.load().mgb_sm_count()


# ---------------------------------------------------------------------------------------------
# F2: stitch  (reference src/magnify/stitch.py:7-46)
# ---------------------------------------------------------------------------------------------
def check_overlap(overlap: int, tile_y: Optional[int] = None, tile_x: Optional[int] = None) -> None:
    """Same exceptions as Stitcher.__init__ (stitch.py:8-9) and __call__ (stitch.py:16-20)."""
    if overlap < 0:
        raise ValueError("Overlap must be non-negative.")
    if tile_y is not None and (overlap >= tile_y or overlap >= tile_x):
        raise ValueError(f"Overlap ({overlap}) must be smaller than tile size ({tile_y}x{tile_x}).")


def stitched_shape(tile_shape: Sequence[int], overlap: int):
    c, t, r, cc, h, w = tile_shape
    return (c, t, r * (h - overlap), cc * (w - overlap))


def alloc_image(shape: Sequence[int], dtype, device) -> torch.Tensor:
    """(C,T,Him,Wim) image whose rows start on 16-byte boundaries: a view `[..., :Wim]` of a buffer
    padded along x.  The vectorised stitch and the staged gather need aligned rows; padding the
    pitch keeps them usable for any tile grid (10x10 tiles at overlap 102 give Wim = 19460, not a
    multiple of 8).  Dense (`is_contiguous()`) whenever Wim already is aligned."""
    c, t, him, wim = (int(v) for v in shape)
    itemsize = torch.empty(0, dtype=dtype).element_size()
    quantum = max(1, 16 // itemsize)
    pitch = -(-wim // quantum) * quantum
    buf = torch.empty((c, t, him, pitch), dtype=dtype, device=device)
    return buf[..., :wim] if pitch != wim else buf


def image_pitch(image: torch.Tensor) -> int:
    """Row pitch (elements) of a dense or x-padded (C,T,H,W) image; raises for other layouts."""
    if image.dim() != 4 or not image.is_cuda:
        raise ValueError("image must be a 4-d CUDA tensor (C,T,H,W)")
    c, t, h, w = image.shape
    if image.numel() == 0:
        return int(w)
    pitch = int(image.stride(2)) if (h > 1 or image.stride(2) >= w) else int(w)
    ok = image.stride(3) == 1 and pitch >= w
    ok = ok and (t == 1 or image.stride(1) == h * pitch) and (c == 1 or image.stride(0) == t * h * pitch)
    if not ok:
        raise ValueError(f"image must be dense or padded along x only, got strides {tuple(image.stride())}")
    return pitch


def to_host_dense(image: torch.Tensor, out: Optional[torch.Tensor] = None, non_blocking: bool = True) -> torch.Tensor:
    """Copy a dense or x-padded device image into a dense (pinned) host tensor with one pitched
    copy on the current stream (no intermediate contiguous device copy)."""
    pitch = image_pitch(image)
    if out is None:
        out = torch.empty(tuple(image.shape), dtype=image.dtype, pin_memory=True)
    if tuple(out.shape) != tuple(image.shape) or out.dtype != image.dtype or not out.is_contiguous():
        raise ValueError("out must be a dense host tensor with the image's shape and dtype")
    c, t, h, w = image.shape
    if pitch == w:
        out.copy_(image, non_blocking=non_blocking)
        return out
    es = image.element_size()
    with torch.cuda.device(image.device):
        _lib.call("mgb_copy2d_async", ctypes.c_void_p(out.data_ptr()), w * es, _ptr(image), pitch * es, w * es,
                  c * t * h, 2, _stream())
    if not non_blocking:
        torch.cuda.current_stream(image.device).synchronize()
    return out


def _image_out(out: Optional[torch.Tensor], shape, dtype, device) -> torch.Tensor:
    if out is None:
        return alloc_image(shape, dtype, device)
    if not isinstance(out, torch.Tensor) or not out.is_cuda or out.dtype != dtype:
        raise TypeError(f"out must be a CUDA tensor of dtype {dtype}")
    if tuple(out.shape) != tuple(shape):
        raise ValueError(f"out has shape {tuple(out.shape)}, expected {tuple(shape)}")
    image_pitch(out)   # validates the layout
    return out


def stitch(tiles: torch.Tensor, overlap: int = 102, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """(C,T,R,Cc,H,W) -> (C,T,R*(H-ov),Cc*(W-ov)); pure copy for any 1/2/4/8-byte dtype.  The result
    is dense or padded along x (see `alloc_image`); `.contiguous()` / `to_host_dense` densify it."""
    _check(tiles, "tiles", ndim=6)
    c, t, r, cc, h, w = tiles.shape
    check_overlap(overlap, h, w)
    out = _image_out(out, stitched_shape(tiles.shape, overlap), tiles.dtype, tiles.device)
    with torch.cuda.device(tiles.device):
        _lib.call("mgb_stitch", _ptr(tiles), _ptr(out), image_pitch(out), c, t, r, cc, h, w, int(overlap),
                  tiles.element_size(), None, _stream())
    return out


# ---------------------------------------------------------------------------------------------
# F1: flat-field  (reference src/magnify/preprocess.py:62-88)
# ---------------------------------------------------------------------------------------------
def _as_table(value, name: str, tile_shape, device) -> torch.Tensor:
    """Expand a scalar / ndarray operand to a float64 (K,H,W) table following NumPy broadcasting
    of `tile - value` on the trailing dims (preprocess.py:83,85).  Only operands that are constant
    over time and tile position are supported (K = 1 shared, or K = C per channel)."""
    c, t, r, cc, h, w = tile_shape
    if isinstance(value, torch.Tensor):
        arr = value.detach().to("cpu").numpy()
    else:
        arr = np.asarray(value)
    arr = arr.astype(np.float64, copy=False)
    if arr.ndim > 6:
        raise ValueError(f"{name} has too many dimensions: {arr.shape}")
    full = arr.reshape((1,) * (6 - arr.ndim) + arr.shape)
    try:
        np.broadcast_shapes(full.shape, tuple(tile_shape))
    except ValueError as e:
        raise ValueError(f"{name} with shape {arr.shape} does not broadcast against tiles {tuple(tile_shape)}") from e
    if full.shape[1] != 1 or full.shape[2] != 1 or full.shape[3] != 1:
        raise NotImplementedError(f"{name} varying over time or tile position is not supported (shape {arr.shape})")
    k = full.shape[0]
    table = np.broadcast_to(full[:, 0, 0, 0], (k, h, w))
    return torch.from_numpy(np.array(table, dtype=np.float64, order="C")).to(device)


class FlatFieldPlan:
    """Device-resident flat/dark tables (float64, (K,H,W)) plus the fast-path coefficients."""

    def __init__(self, tile_shape, flatfield=1.0, darkfield=0.0, device="cuda"):
        self.tile_shape = tuple(int(s) for s in tile_shape)
        c = self.tile_shape[0]
        self.identity = (
            np.isscalar(flatfield) and np.isscalar(darkfield) and float(flatfield) == 1.0 and float(darkfield) == 0.0
        )
        flat = _as_table(flatfield, "flatfield", self.tile_shape, device)
        dark = _as_table(darkfield, "darkfield", self.tile_shape, device)
        k = max(flat.shape[0], dark.shape[0])
        if k not in (1, c):
            raise ValueError("flatfield/darkfield leading dimension must be 1 or the channel count")
        if flat.shape[0] != k:
            flat = flat.expand(k, -1, -1).contiguous()
        if dark.shape[0] != k:
            dark = dark.expand(k, -1, -1).contiguous()
        # The reference would silently produce inf/nan for flat <= 0 (undefined cast at
        # preprocess.py:87); reject it instead.
        if not bool(torch.isfinite(flat).all()) or not bool((flat > 0).all()):
            raise ValueError("flatfield must be finite and strictly positive")
        if not bool(torch.isfinite(dark).all()):
            raise ValueError("darkfield must be finite")
        self.k = int(k)
        self.flat, self.dark = flat, dark
        self.gain = torch.empty_like(flat)
        self.bias = torch.empty_like(flat)
        self.maxima = torch.zeros(2, dtype=torch.float64, device=device)
        self._workspace = None

    def workspace(self, nbytes: int, device) -> torch.Tensor:
        if self._workspace is None or self._workspace.numel() < nbytes:
            self._workspace = torch.empty(nbytes, dtype=torch.uint8, device=device)
        return self._workspace


def flatfield_maxima(tiles: torch.Tensor, plan: FlatFieldPlan) -> torch.Tensor:
    """Pass 1: the two global maxima (M, M2) of preprocess.py:84,86 over this rank's tiles, as a
    float64[2] device tensor (plan.maxima).  Multi-GPU callers all-reduce it with MAX."""
    _check(tiles, "tiles", ndim=6)
    c, t, r, cc, h, w = tiles.shape
    planes, hw = t * r * cc, h * w
    with torch.cuda.device(tiles.device):
        plan.maxima.zero_()
        if tiles.numel() == 0:
            return plan.maxima
        if tiles.dtype == torch.uint16 and hw % 8 == 0 and tiles.data_ptr() % 16 == 0:
            base = -(-(hw // 8) // 256) * plan.k
            n_planes = c * planes if plan.k == 1 else planes
            splits = max(1, min(n_planes // 8 if n_planes >= 16 else 1, -(-sm_count() * 16 // base), 4096))
            ws = plan.workspace(splits * plan.k * hw * 2, tiles.device)
            _lib.call("mgb_flatfield_tilemax_u16", _ptr(tiles), c, planes, hw, plan.k, splits, _ptr(ws), _stream())
            _lib.call("mgb_flatfield_maxima", _ptr(ws), splits, plan.k, hw, _ptr(plan.flat), _ptr(plan.dark),
                      _ptr(plan.maxima), _stream())
        else:
            if tiles.dtype not in _DTYPE_CODE:
                raise TypeError(f"flat-field supports uint8/uint16/float32/float64 tiles, got {tiles.dtype}")
            _lib.call("mgb_flatfield_maxima_generic", _ptr(tiles), _DTYPE_CODE[tiles.dtype], c, planes, hw, plan.k,
                      _ptr(plan.flat), _ptr(plan.dark), _ptr(plan.maxima), _stream())
    return plan.maxima


def flatfield_maxima_accumulate(block: torch.Tensor, plan: FlatFieldPlan, channel: int) -> None:
    """Pass 1 on one contiguous block of tiles of one channel (any leading shape, trailing
    (H, W)), accumulating into plan.maxima (which the caller zeroed).  Used by the staging
    loop, where each (channel, timepoint) block arrives separately."""
    _check(block, "block")
    h, w = block.shape[-2:]
    hw = h * w
    planes = block.numel() // hw
    if planes == 0:
        return
    k_off = (channel if plan.k > 1 else 0) * hw
    flat = plan.flat.view(-1)[k_off:k_off + hw]
    dark = plan.dark.view(-1)[k_off:k_off + hw]
    with torch.cuda.device(block.device):
        if block.dtype == torch.uint16 and hw % 8 == 0 and block.data_ptr() % 16 == 0:
            base = -(-(hw // 8) // 256)
            splits = max(1, min(planes // 8 if planes >= 16 else 1, -(-sm_count() * 16 // base), 4096))
            ws = plan.workspace(splits * hw * 2, block.device)
            _lib.call("mgb_flatfield_tilemax_u16", _ptr(block), 1, planes, hw, 1, splits, _ptr(ws), _stream())
            _lib.call("mgb_flatfield_maxima", _ptr(ws), splits, 1, hw, _ptr(flat), _ptr(dark), _ptr(plan.maxima),
                      _stream())
        else:
            if block.dtype not in _DTYPE_CODE:
                raise TypeError(f"flat-field supports uint8/uint16/float32/float64 tiles, got {block.dtype}")
            _lib.call("mgb_flatfield_maxima_generic", _ptr(block), _DTYPE_CODE[block.dtype], 1, planes, hw, 1,
                      _ptr(flat), _ptr(dark), _ptr(plan.maxima), _stream())


def flatfield_stitch(
    tiles: torch.Tensor,
    flatfield=1.0,
    darkfield=0.0,
    overlap: int = 102,
    plan: Optional[FlatFieldPlan] = None,
    maxima: Optional[torch.Tensor] = None,
    group=None,
    out: Optional[torch.Tensor] = None,
) -> torch.Tensor:
    """flatfield_correct (preprocess.py:83-87) followed by stitch (stitch.py:22-39), fused.

    maxima: precomputed (M, M2) float64[2] device tensor (already global); when None they are
    computed here and, if `group` is a torch.distributed process group, all-reduced with MAX
    (both maxima are global over channel x time x tiles, SURVEY.md section 0 fact 9)."""
    _check(tiles, "tiles", ndim=6)
    c, t, r, cc, h, w = tiles.shape
    check_overlap(overlap, h, w)
    if plan is None:
        plan = FlatFieldPlan(tiles.shape, flatfield, darkfield, device=tiles.device)
    if plan.identity and tiles.dtype in _UNSIGNED:
        # (x * M) / M == x exactly for non-negative integers below 2^53: the defaults are the identity.
        # Float tiles still go through the arithmetic (clip(min=0) zeroes negatives, preprocess.py:83).
        return stitch(tiles, overlap, out=out)
    out = _image_out(out, stitched_shape(tiles.shape, overlap), tiles.dtype, tiles.device)
    if tiles.numel() == 0:
        return out
    with torch.cuda.device(tiles.device):
        if maxima is None:
            maxima = flatfield_maxima(tiles, plan)
            if group is not None:
                import torch.distributed as dist

                dist.all_reduce(maxima, op=dist.ReduceOp.MAX, group=group)
        else:
            _check(maxima, "maxima", dtype=torch.float64)
            if maxima.data_ptr() != plan.maxima.data_ptr():
                plan.maxima.copy_(maxima)
            maxima = plan.maxima
        rc = _lib.MGB_EALIGN
        if tiles.dtype == torch.uint16:
            _lib.call("mgb_flatfield_tables", _ptr(plan.flat), _ptr(plan.dark), plan.k, h * w, _ptr(maxima),
                      _ptr(plan.gain), _ptr(plan.bias), _stream())
            rc = _lib.try_call("mgb_flatfield_stitch_u16", _ptr(tiles), _ptr(out), image_pitch(out), c, t, r, cc, h, w,
                               int(overlap),
                               plan.k, _ptr(plan.flat), _ptr(plan.dark), _ptr(plan.gain), _ptr(plan.bias),
                               _ptr(maxima), _stream())
            if rc not in (0, _lib.MGB_EALIGN):
                raise _lib.MagnifyB200Error("mgb_flatfield_stitch_u16", rc, _lib.error_string(rc))
        if rc == _lib.MGB_EALIGN:
            if tiles.dtype not in _DTYPE_CODE:
                raise TypeError(f"flat-field supports uint8/uint16/float32/float64 tiles, got {tiles.dtype}")
            tmp = torch.empty_like(tiles)
            _lib.call("mgb_flatfield_apply_generic", _ptr(tiles), _ptr(tmp), _DTYPE_CODE[tiles.dtype], c, t * r * cc,
                      h * w, plan.k, _ptr(plan.flat), _ptr(plan.dark), _ptr(maxima), _stream())
            stitch(tmp, overlap, out=out)
    return out


def flatfield_correct(tiles: torch.Tensor, flatfield=1.0, darkfield=0.0, plan=None, maxima=None, group=None):
    """flatfield_correct alone (preprocess.py:83-87): corrected tiles in tile layout."""
    _check(tiles, "tiles", ndim=6)
    c, t, r, cc, h, w = tiles.shape
    if plan is None:
        plan = FlatFieldPlan(tiles.shape, flatfield, darkfield, device=tiles.device)
    if plan.identity and tiles.dtype in _UNSIGNED:
        return tiles.clone()
    # Every tile is its own 1x1 "image": same kernel, overlap 0.
    as_images = tiles.view(c, t * r * cc, 1, 1, h, w)
    plan_shape = plan.tile_shape
    dense = torch.empty((c, t * r * cc, h, w), dtype=tiles.dtype, device=tiles.device)   # tile layout is dense
    out = flatfield_stitch(as_images, overlap=0, plan=plan, maxima=maxima, group=group, out=dense)
    plan.tile_shape = plan_shape
    return out.view(tiles.shape)


# ---------------------------------------------------------------------------------------------
# F3: bounding boxes  (reference src/magnify/utils.py:55-80)
# ---------------------------------------------------------------------------------------------
def bounding_boxes(x: torch.Tensor, y: torch.Tensor, roi_length: int, im_x: int, im_y: int, want_rel: bool = False):
    """boxes[..., :] = (top, left) of bounding_box(round(x), round(y), L, im_x, im_y); optional
    rel[..., :] = (round(y) - top, round(x) - left) (find.py:380-381).  x, y float64, any shape."""
    _check(x, "x", dtype=torch.float64)
    _check(y, "y", dtype=torch.float64)
    if x.shape != y.shape:
        raise ValueError("x and y must have the same shape")
    if im_x < roi_length or im_y < roi_length:
        raise ValueError(f"image ({im_y}x{im_x}) is smaller than roi_length {roi_length}")
    boxes = torch.empty(tuple(x.shape) + (2,), dtype=torch.int32, device=x.device)
    rel = torch.empty_like(boxes) if want_rel else None
    with torch.cuda.device(x.device):
        _lib.call("mgb_bounding_boxes", _ptr(x), _ptr(y), x.numel(), int(roi_length), int(im_x), int(im_y),
                  _ptr(boxes), _ptr(rel), _stream())
    return (boxes, rel) if want_rel else boxes


# ---------------------------------------------------------------------------------------------
# F4 + R: ROI gather and masked reductions
# ---------------------------------------------------------------------------------------------
def _check_boxes(boxes, m, t):
    _check(boxes, "boxes", dtype=torch.int32, ndim=3)
    if tuple(boxes.shape) != (m, t, 2):
        raise ValueError(f"boxes must have shape ({m}, {t}, 2), got {tuple(boxes.shape)}")


def spatial_order(boxes: torch.Tensor, band: int = 32) -> torch.Tensor:
    """Permutation of the markers sorted by (top // band, left) of their first box: markers that
    are processed together then read neighbouring image rows, so DRAM lines shared by nearby or
    overlapping windows are fetched once and hit in L2 afterwards.  boxes (M,T,2) or (M,2)."""
    b = boxes[:, 0] if boxes.dim() == 3 else boxes
    if b.shape[0] == 0:
        return torch.zeros(0, dtype=torch.int32, device=boxes.device)
    key = (b[:, 0].to(torch.int64) // band) * (1 << 32) + b[:, 1].to(torch.int64)
    return torch.argsort(key).to(torch.int32).contiguous()


def _check_order(order, m):
    if order is None:
        return None
    _check(order, "order", dtype=torch.int32, ndim=1)
    if order.numel() != m:
        raise ValueError("order must be a permutation of the markers")
    return order


def roi_gather(image: torch.Tensor, boxes: torch.Tensor, roi_length: int, out: Optional[torch.Tensor] = None,
               order: Optional[torch.Tensor] = None):
    """roi[m,c,t] = image[c,t, top:top+L, left:left+L]  (find.py:160-169,324-334,589-602)."""
    pitch = image_pitch(image)
    c, t, h, w = image.shape
    m = boxes.shape[0]
    _check_boxes(boxes, m, t)
    shape = (m, c, t, roi_length, roi_length)
    if out is None:
        out = torch.empty(shape, dtype=image.dtype, device=image.device)
    elif tuple(out.shape) != shape or out.dtype != image.dtype:
        raise ValueError(f"out must have shape {shape} and dtype {image.dtype}")
    elif not out.is_contiguous():
        raise ValueError("out must be contiguous")   # the kernels write roi + n*L*L densely
    with torch.cuda.device(image.device):
        _lib.call("mgb_roi_gather", _ptr(image), pitch, c, t, h, w, image.element_size(), _ptr(boxes),
                  _ptr(_check_order(order, m)), m, int(roi_length), _ptr(out), _stream())
    return out


def _masks_u8(fg, bg, m, roi_length):
    fg = fg.view(torch.uint8) if fg.dtype == torch.bool else fg
    bg = bg.view(torch.uint8) if bg.dtype == torch.bool else bg
    _check(fg, "fg", dtype=torch.uint8, ndim=4)
    _check(bg, "bg", dtype=torch.uint8, ndim=4)
    tm = fg.shape[1]
    if tuple(fg.shape) != (m, tm, roi_length, roi_length) or fg.shape != bg.shape:
        raise ValueError(f"fg/bg must have shape ({m}, Tm, {roi_length}, {roi_length})")
    return fg, bg, tm


def _default_mask_t(mask_t, tm, t, device, what="fg/bg"):
    if mask_t is None:
        if tm == 1:
            mask_t = torch.zeros(t, dtype=torch.int32, device=device)
        elif tm == t:
            mask_t = torch.arange(t, dtype=torch.int32, device=device)
        else:
            raise ValueError(f"mask_t is required when {what} hold neither 1 nor T timesteps")
    _check(mask_t, "mask_t", dtype=torch.int32, ndim=1)
    if mask_t.numel() != t:
        raise ValueError("mask_t must have one entry per timepoint")
    return mask_t


def mask_count_max(fg: torch.Tensor, bg: torch.Tensor):
    """(largest fg pixel count, largest bg pixel count) over all masks of (M,Tm,L,L) stacks, as
    Python ints (one small kernel + a 8-byte read-back).  The fused gather sizes its per-marker
    value lists from these bounds; callers that reuse masks (a `QuantifyPlan`) compute them once."""
    fg = fg.view(torch.uint8) if fg.dtype == torch.bool else fg
    bg = bg.view(torch.uint8) if bg.dtype == torch.bool else bg
    _check(fg, "fg", dtype=torch.uint8)
    _check(bg, "bg", dtype=torch.uint8)
    if fg.shape != bg.shape or fg.dim() < 2:
        raise ValueError("fg and bg must have the same shape (..., L, L)")
    length = fg.shape[-1] * fg.shape[-2]
    n = fg.numel() // length if length else 0
    counts = torch.empty(2, dtype=torch.int32, device=fg.device)
    with torch.cuda.device(fg.device):
        _lib.call("mgb_mask_count_max", _ptr(fg), _ptr(bg), n, length, _ptr(counts), _stream())
    c = counts.cpu()
    return int(c[0]), int(c[1])


last_gather_fused = True   # diagnostic: did the last roi_gather_stats call get its medians from the fused kernel?


def roi_gather_stats(
    image: torch.Tensor,
    boxes: torch.Tensor,
    fg: torch.Tensor,
    bg: torch.Tensor,
    roi_length: int,
    mask_t: Optional[torch.Tensor] = None,
    want_roi: bool = True,
    out_roi: Optional[torch.Tensor] = None,
    out_stats: Optional[torch.Tensor] = None,
    order: Optional[torch.Tensor] = None,
    peer_stats: Optional[Sequence[int]] = None,
    medians: bool = True,
    mask_counts: Optional[Sequence[int]] = None,
):
    """Gather fused with per-(marker, channel, time) masked counts / sums / means / medians.

    fg, bg: (M, Tm, L, L) uint8 (any non-zero byte = set) or bool; mask_t (T,) int32 maps
    timepoints to mask timesteps (default: all 0 when Tm == 1, identity when Tm == T).  Returns
    (roi | None, stats) with stats (M,C,T,8) float64 in `STATS` order; with medians=False the two
    median columns are NaN.

    mask_counts: `mask_count_max(fg, bg)` when the caller already has it (otherwise it is computed
    here, which costs a device->host read of 8 bytes).  Masks of at most 1024 fg / 2560 bg pixels
    per marker get sums and medians from the staged window in one pass; larger masks take the
    dp2a sums and a separate exact-median pass over the crops (peer_stats: medians stay NaN)."""
    if image.dtype != torch.uint16:
        raise TypeError(f"image must have dtype torch.uint16, got {image.dtype}")
    pitch = image_pitch(image)
    c, t, h, w = image.shape
    m = boxes.shape[0]
    _check_boxes(boxes, m, t)
    fg, bg, tm = _masks_u8(fg, bg, m, roi_length)
    mask_t = _default_mask_t(mask_t, tm, t, image.device)
    roi = None
    shape = (m, c, t, roi_length, roi_length)
    if want_roi:
        roi = out_roi if out_roi is not None else torch.empty(shape, dtype=image.dtype, device=image.device)
        if tuple(roi.shape) != shape or roi.dtype != image.dtype:
            raise ValueError(f"out_roi must have shape {shape} and dtype {image.dtype}")
        if not roi.is_contiguous():
            raise ValueError("out_roi must be contiguous")   # the kernels write roi + n*L*L densely
    # the staged kernels store each 64-byte summary record as four 16-byte vectors
    if peer_stats is not None:
        if any(int(a) % 16 for a in peer_stats):
            raise ValueError("every peer_stats address must be 16-byte aligned")
    else:
        stats = out_stats if out_stats is not None else torch.empty((m, c, t, NSTATS), dtype=torch.float64,
                                                                    device=image.device)
        if tuple(stats.shape) != (m, c, t, NSTATS) or stats.dtype != torch.float64 or not stats.is_contiguous():
            raise ValueError(f"out_stats must be contiguous float64 with shape (M, C, T, {NSTATS})")
        if stats.data_ptr() % 16:
            raise ValueError("out_stats must be 16-byte aligned")
    if mask_counts is None:
        mask_counts = mask_count_max(fg, bg) if m * tm > 0 else (0, 0)
    nf_max, nb_max = int(mask_counts[0]), int(mask_counts[1])
    done = ctypes.c_int(0)
    if peer_stats is not None:
        # Multi-GPU: the kernel writes every summary record into this rank's block of each rank's
        # gathered buffer (peer-mapped addresses, see magnify_b200.dist.SymmetricSummaries).
        n_peers = len(peer_stats)
        arr = (ctypes.c_uint64 * n_peers)(*[int(a) for a in peer_stats])
        with torch.cuda.device(image.device):
            _lib.call("mgb_roi_gather_stats_peers_u16", _ptr(image), pitch, c, t, h, w, _ptr(boxes),
                      _ptr(_check_order(order, m)), _ptr(mask_t), tm, _ptr(fg), _ptr(bg), m, int(roi_length),
                      _ptr(roi), arr, n_peers, int(bool(medians)), nf_max, nb_max, ctypes.byref(done), _stream())
        if medians and not done.value and m * c * t > 0:
            raise RuntimeError("peer_stats needs the fused gather (masks of at most 1024 fg / 2560 bg pixels per marker, "
                               "uint16 image); gather locally and all_gather the summaries instead")
        return roi, None
    with torch.cuda.device(image.device):
        _lib.call("mgb_roi_gather_stats_u16", _ptr(image), pitch, c, t, h, w, _ptr(boxes), _ptr(_check_order(order, m)),
                  _ptr(mask_t), tm, _ptr(fg), _ptr(bg), m, int(roi_length), _ptr(roi), _ptr(stats),
                  int(bool(medians)), nf_max, nb_max, ctypes.byref(done), _stream())
    global last_gather_fused
    last_gather_fused = bool(done.value) or not medians
    if medians and not done.value and m * c * t > 0:
        # masks too large for the in-kernel lists (or an image the staged kernels do not take):
        # exact medians from the crops in a second pass
        crops = roi if roi is not None else roi_gather(image, boxes, roi_length, order=order)
        _median_into(crops, fg, mask_t, tm, stats, 6)
        _median_into(crops, bg, mask_t, tm, stats, 7)
    return roi, stats


def _median_into(roi, mask, mask_t, tm, stats, column: int) -> None:
    m, c, t, length, _ = roi.shape
    out = stats.view(-1)[column:]
    with torch.cuda.device(roi.device):
        _lib.call("mgb_roi_median_u16" if roi.dtype == torch.uint16 else "mgb_roi_median_f32", _ptr(roi), m, c, t,
                  int(length), _ptr(mask_t), tm, _ptr(mask), _ptr(out), NSTATS, _stream())


def roi_stats(roi: torch.Tensor, fg: torch.Tensor, bg: torch.Tensor, mask_t: Optional[torch.Tensor] = None,
              medians: bool = True) -> torch.Tensor:
    """Masked counts / sums / means / medians of an existing roi (M,C,T,L,L) uint16 or float32 ->
    (M,C,T,8) float64 (float32: float64 accumulation, NaN pixels skipped)."""
    if roi.dtype not in (torch.uint16, torch.float32):
        raise TypeError(f"roi must be uint16 or float32, got {roi.dtype}")
    _check(roi, "roi", ndim=5)
    m, c, t, length, _ = roi.shape
    fg, bg, tm = _masks_u8(fg, bg, m, length)
    mask_t = _default_mask_t(mask_t, tm, t, roi.device)
    stats = torch.empty((m, c, t, NSTATS), dtype=torch.float64, device=roi.device)
    with torch.cuda.device(roi.device):
        _lib.call("mgb_roi_stats_u16" if roi.dtype == torch.uint16 else "mgb_roi_stats_f32", _ptr(roi), m, c, t,
                  int(length), _ptr(mask_t), tm, _ptr(fg), _ptr(bg), _ptr(stats), _stream())
    if medians and m * c * t > 0:
        _median_into(roi, fg, mask_t, tm, stats, 6)
        _median_into(roi, bg, mask_t, tm, stats, 7)
    return stats


def roi_median(roi: torch.Tensor, mask: torch.Tensor, mask_t: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Exact masked median per (m,c,t) -> (M,C,T) float64, NaN for an empty mask
    (`roi.where(mask).median(dim=["roi_x","roi_y"])`, identify.py:79, filter.py:21-22); uint16 or
    float32 roi (NaN pixels skipped), any roi_length."""
    if roi.dtype not in (torch.uint16, torch.float32):
        raise TypeError(f"roi must be uint16 or float32, got {roi.dtype}")
    _check(roi, "roi", ndim=5)
    m, c, t, length, _ = roi.shape
    mask = mask.view(torch.uint8) if mask.dtype == torch.bool else mask
    _check(mask, "mask", dtype=torch.uint8, ndim=4)
    tm = mask.shape[1]
    if tuple(mask.shape) != (m, tm, length, length):
        raise ValueError(f"mask must have shape ({m}, Tm, {length}, {length})")
    mask_t = _default_mask_t(mask_t, tm, t, roi.device, "mask")
    out = torch.empty((m, c, t), dtype=torch.float64, device=roi.device)
    with torch.cuda.device(roi.device):
        _lib.call("mgb_roi_median_u16" if roi.dtype == torch.uint16 else "mgb_roi_median_f32", _ptr(roi), m, c, t,
                  int(length), _ptr(mask_t), tm, _ptr(mask), _ptr(out), 1, _stream())
    return out


# ---------------------------------------------------------------------------------------------
# F5-F8: masks
# ---------------------------------------------------------------------------------------------
def chip_masks(rel: torch.Tensor, fg_radius: torch.Tensor, inner_radius: int, outer_radius: int, roi_length: int,
               want_counts: bool = False):
    """fg = disc(fg_radius[m]), bg = annulus(inner < d <= outer) centred on rel[m] = (y_rel, x_rel)
    (utils.py:30-52 via find.py:380-400).  Returns fg, bg (M,L,L) uint8 [, counts (M,2) int32]."""
    _check(rel, "rel", dtype=torch.int32, ndim=2)
    _check(fg_radius, "fg_radius", dtype=torch.int32, ndim=1)
    m = rel.shape[0]
    if rel.shape[1] != 2 or fg_radius.shape[0] != m:
        raise ValueError("rel must be (M,2) and fg_radius (M,)")
    fg = torch.empty((m, roi_length, roi_length), dtype=torch.uint8, device=rel.device)
    bg = torch.empty_like(fg)
    counts = torch.empty((m, 2), dtype=torch.int32, device=rel.device) if want_counts else None
    with torch.cuda.device(rel.device):
        _lib.call("mgb_chip_masks", _ptr(rel), _ptr(fg_radius), int(inner_radius), int(outer_radius), m,
                  int(roi_length), _ptr(fg), _ptr(bg), _ptr(counts), _stream())
    return (fg, bg, counts) if want_counts else (fg, bg)


_HW_CACHE: dict = {}


def disc_halfwidth_table(rmax: int) -> np.ndarray:
    """Host table hw[r, |drow|] of the reference's filled disc (utils.py:398-465) for r = 1..rmax."""
    rmax = int(rmax)
    if rmax in _HW_CACHE:
        return _HW_CACHE[rmax]
    table = np.zeros((rmax + 1, rmax + 1), dtype=np.int32)
    lib = _lib.load()
    for r in range(1, rmax + 1):
        row = (ctypes.c_int32 * (r + 1))()
        rc = lib.mgb_disc_halfwidths(r, row)
        if rc != 0:
            raise _lib.MagnifyB200Error("mgb_disc_halfwidths", rc, _lib.error_string(rc))
        table[r, : r + 1] = np.frombuffer(row, dtype=np.int32)
    _HW_CACHE[rmax] = table
    return table


def _upload_async(values: np.ndarray, device) -> torch.Tensor:
    """Host array -> device on the current stream without blocking the host (pinned staging from
    torch's caching host allocator, which keeps the block until the copy has run)."""
    return torch.from_numpy(np.ascontiguousarray(values)).pin_memory().to(device, non_blocking=True)


def bead_labels(beads, im_y: int, im_x: int, device=None) -> torch.Tensor:
    """Label raster of utils.circle_labels (utils.py:380-395): beads (M,3) int32 rows
    (row, col, radius >= 1) -> (im_y, im_x) int32 with -1 none / i sole owner / -2 shared.

    beads: a device tensor, or a HOST array together with `device` -- then the radius range is
    taken on the host and nothing is read back from the device (a read would wait behind whatever
    download is in flight on the copy engine)."""
    if isinstance(beads, np.ndarray):
        if device is None:
            raise ValueError("device is required with host beads")
        host = np.ascontiguousarray(beads, dtype=np.int32)
        if host.ndim != 2 or (host.shape[0] and host.shape[1] != 3):
            raise ValueError("beads must be (M,3)")
        m = host.shape[0]
        rmin, rmax = (int(host[:, 2].min()), int(host[:, 2].max())) if m else (1, 0)
        beads = _upload_async(host, torch.device(device))
    else:
        _check(beads, "beads", dtype=torch.int32, ndim=2)
        m = beads.shape[0]
        if m and beads.shape[1] != 3:
            raise ValueError("beads must be (M,3)")
        rmin, rmax = (int(beads[:, 2].min().item()), int(beads[:, 2].max().item())) if m else (1, 0)
    if m and rmin < 1:
        raise ValueError("bead radii must be >= 1 (filled_circle_points(0) raises in the reference)")
    labels = torch.empty((im_y, im_x), dtype=torch.int32, device=beads.device)
    hw = _upload_async(disc_halfwidth_table(max(rmax, 1)), beads.device)
    with torch.cuda.device(beads.device):
        _lib.call("mgb_bead_labels", _ptr(beads), m, int(im_y), int(im_x), _ptr(hw), max(rmax, 1), _ptr(labels),
                  _stream())
    return labels


def bead_masks(labels: torch.Tensor, boxes: torch.Tensor, roi_length: int, want_counts: bool = False):
    """fg[m] = labels[box m] == m, bg[m] = labels[box m] == -1 (find.py:580-584); boxes (M,2)."""
    _check(labels, "labels", dtype=torch.int32, ndim=2)
    _check(boxes, "boxes", dtype=torch.int32, ndim=2)
    m = boxes.shape[0]
    h, w = labels.shape
    fg = torch.empty((m, roi_length, roi_length), dtype=torch.uint8, device=labels.device)
    bg = torch.empty_like(fg)
    counts = torch.empty((m, 2), dtype=torch.int32, device=labels.device) if want_counts else None
    with torch.cuda.device(labels.device):
        _lib.call("mgb_bead_masks", _ptr(labels), h, w, _ptr(boxes), m, int(roi_length), _ptr(fg), _ptr(bg),
                  _ptr(counts), _stream())
    return (fg, bg, counts) if want_counts else (fg, bg)


# ---------------------------------------------------------------------------------------------
# filter_nonround  (reference src/magnify/filter.py:40-62)
# ---------------------------------------------------------------------------------------------
def mask_perimeters(masks: torch.Tensor) -> torch.Tensor:
    """Perimeter of every (L, L) mask of a (M, L, L) uint8 / bool stack as
    `sum(cv.arcLength(c, True) for c in cv.findContours(mask, RETR_EXTERNAL, CHAIN_APPROX_SIMPLE)[0])`
    measures it (filter.py:54-55); float64 (M,)."""
    masks = masks.view(torch.uint8) if masks.dtype == torch.bool else masks
    _check(masks, "masks", dtype=torch.uint8, ndim=3)
    m, length, width = masks.shape
    if length != width:
        raise ValueError("masks must be square (M, L, L)")
    out = torch.empty(m, dtype=torch.float64, device=masks.device)
    with torch.cuda.device(masks.device):
        _lib.call("mgb_mask_perimeters", _ptr(masks), m, length, _ptr(out), _stream())
    return out
