"""Masked per-marker reductions the reference's consumers run on roi/fg/bg.

TEST INFRASTRUCTURE (see oracle/__init__.py).  PARITY UNPINNED by the reference's suite (no
test asserts an intensity).  The reference expressions are xarray's
`roi.where(fg).mean(dim=["roi_x","roi_y"])` / `.median(...)` / `fg.sum(...)`
(src/magnify/identify.py:76-80, filter.py:21-22,51,74,82, README.md:21-22): `where` fills
masked-out pixels with NaN and the reductions skip NaN (nanmean / nanmedian), so an empty
mask yields NaN.  Restated here in float64, except the medians of a float roi: `where` keeps a
float32 roi float32, and np.nanmedian averages the two middle values of a float32 array in float32
(the sum rounded to float32, inf where it overflows, then halved).  Integer rois are widened by
`where`; the half-sum of two 16-bit values is exact in any float type, so their medians are taken
in float64.  (For fewer than 600 pixels per window np.nanmedian takes a masked-array path that also
"averages" an odd count's single middle value with itself, so a float32 middle value above half the
float32 maximum becomes inf there; the kernels return the middle value, as np.median does.)
"""
from __future__ import annotations

import warnings

import numpy as np

def _median_values(roi: np.ndarray) -> np.ndarray:
    """roi in the dtype `roi.where(mask)` reduces its median in (see the module docstring)."""
    return roi if np.issubdtype(roi.dtype, np.floating) else roi.astype(np.float64)


STATS = ("n_fg", "n_bg", "sum_fg", "sum_bg", "mean_fg", "mean_bg", "median_fg", "median_bg")


def masked_stats(roi: np.ndarray, fg: np.ndarray, bg: np.ndarray) -> np.ndarray:
    """roi (M, C, T, L, L), fg/bg (M, T, L, L) bool -> (M, C, T, 8) float64 in STATS order."""
    m, c, t = roi.shape[:3]
    out = np.empty((m, c, t, len(STATS)), dtype=np.float64)
    r = roi.astype(np.float64)
    rm = _median_values(roi)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)
        for k, mask in enumerate((fg, bg)):
            mk = np.broadcast_to(mask[:, None], r.shape)
            vals = np.where(mk, r, np.nan)
            out[..., 0 + k] = np.broadcast_to(mask.sum(axis=(-2, -1))[:, None], (m, c, t))
            out[..., 2 + k] = np.nansum(vals, axis=(-2, -1))
            out[..., 4 + k] = np.nanmean(vals, axis=(-2, -1))
            med = np.where(mk, rm, rm.dtype.type(np.nan))
            out[..., 6 + k] = np.nanmedian(med.reshape(med.shape[:3] + (-1,)), axis=-1)
    return out


def masked_median(roi: np.ndarray, mask: np.ndarray) -> np.ndarray:
    """`roi.where(mask).median(dim=["roi_x","roi_y"])` -> (M, C, T) float64 (NaN when empty)."""
    r = _median_values(roi)
    vals = np.where(np.broadcast_to(mask[:, None], r.shape), r, r.dtype.type(np.nan))
    flat = vals.reshape(vals.shape[:3] + (-1,))
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)
        return np.nanmedian(flat, axis=-1).astype(np.float64)


def mrbles_intensities(roi: np.ndarray, fg: np.ndarray, bg: np.ndarray) -> np.ndarray:
    """identify.py:76-80 at time 0: `sel.where(sel.fg).mean(...) - sel.where(sel.bg).median(...)`.
    roi (M,C,T,L,L), fg/bg (M,T,L,L) -> (M,C)."""
    r0, f0, b0 = roi[:, :, :1], fg[:, :1], bg[:, :1]
    return masked_stats(r0, f0, b0)[:, :, 0, 4] - masked_median(r0, b0)[:, :, 0]


def filter_expression_valid(roi: np.ndarray, fg: np.ndarray, bg: np.ndarray, valid: np.ndarray, channels,
                            min_contrast=None) -> np.ndarray:
    """filter.py:11-37: per search channel, medians of fg and bg at time 0; markers whose fg-bg
    exceeds 4 standard deviations of all pairwise background differences (or `min_contrast`) are
    expressed; `valid &= any-channel-expressed`.  valid (M,T) bool; channels = channel indices."""
    expressed = np.zeros(valid.shape, dtype=bool)
    for c in channels:
        r0 = roi[:, c : c + 1, :1]
        fgm = masked_median(r0, fg[:, :1])[:, 0, 0]
        bgm = masked_median(r0, bg[:, :1])[:, 0, 0]
        if min_contrast is None:
            diffs = bgm[:, np.newaxis] - bgm[np.newaxis, :]          # :26-29
            offdiag = np.ones_like(diffs, dtype=bool) & (~np.eye(len(diffs), dtype=bool))
            upper = 4 * diffs[offdiag].std()                          # :32
        else:
            upper = min_contrast
        expressed |= (fgm - bgm > upper)[:, None]                     # :35 (broadcast over time)
    return valid & expressed


def filter_leaky_valid(roi: np.ndarray, fg: np.ndarray, bg: np.ndarray, valid: np.ndarray, tag: np.ndarray,
                       mark_row: np.ndarray, channels) -> np.ndarray:
    """filter.py:65-94: a tagged marker next (in stacked mark order) to an untagged ("" tag) one
    stays valid only if that blank neighbour is "empty": its fg-bg median contrast at time 0 is
    below 5 standard deviations of all pairwise background differences.  Neighbours are i-1 (when
    the marker's row > 0) and i+1 (when its row < max row), exactly as the reference indexes them.
    valid (M,T) bool, tag (M,) str, mark_row (M,) int; channels = channel indices."""
    valid = valid.copy()
    m = roi.shape[0]
    for c in channels:
        r0 = roi[:, c : c + 1, :1]
        bgm = masked_median(r0, bg[:, :1])[:, 0, 0]
        fgm = masked_median(r0, fg[:, :1])[:, 0, 0]
        diffs = bgm[:, np.newaxis] - bgm[np.newaxis, :]              # :76-79
        offdiag = np.ones_like(diffs, dtype=bool) & (~np.eye(len(diffs), dtype=bool))
        upper = 5 * diffs[offdiag].std()                              # :82
        empty = fgm - bgm < upper                                     # :84
        for i in range(m):                                            # :85-92
            if tag[i] == "":
                continue
            if mark_row[i] > 0 and tag[i - 1] == "":
                valid[i] &= empty[i - 1]
            if mark_row[i] < mark_row.max() and tag[i + 1] == "":
                valid[i] &= empty[i + 1]
    return valid


def filter_nonround_valid(fg: np.ndarray, valid: np.ndarray, min_roundness: float = 0.75) -> np.ndarray:
    """filter.py:40-62 with the reference's own OpenCV calls (cv2 is in the image): per marker,
    external contours of the time-0 foreground, perimeter = sum of closed arc lengths, invalid
    when there is no contour or 4 pi area / perimeter^2 <= min_roundness.  fg (M,T,L,L), valid (M,T)."""
    import cv2 as cv

    valid = valid.copy()
    masks = (fg[:, 0] != 0).astype(np.uint8) * 255                  # utils.to_uint8 of a boolean stack
    areas = fg[:, 0].sum(axis=(1, 2))
    for i in range(len(masks)):
        contours, _ = cv.findContours(masks[i], cv.RETR_EXTERNAL, cv.CHAIN_APPROX_SIMPLE)   # :54
        perimeter = sum(cv.arcLength(c, True) for c in contours)                             # :55
        if perimeter == 0:
            valid[i] = False                                                                  # :56-58
            continue
        valid[i] &= 4 * np.pi * float(areas[i]) / perimeter**2 > min_roundness               # :59-60
    return valid
