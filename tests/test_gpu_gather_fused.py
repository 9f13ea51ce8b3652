"""Every configuration of the fused ROI gather (roi_lists.cu) against the float64 oracle.

The host launcher of the fused gather picks one of many compiled kernels: the crop copy loop
(by L, L % 8 and the alignment of the crop buffer), one CTA or one warp per marker, the warps
per CTA and stages per warp that fit in shared memory, the list capacities, the split of the
last wave.  Each case here states which configuration it expects (`launch_plan`, `copy_class`
restate the launcher's host logic), asserts that the fused kernel ran or did not run
(`ops.last_gather_fused`), and compares crops, counts, sums, means and medians with
`oracle.rois.gather_rois` / `oracle.reduce` exactly (means to 1e-12 relative).

The argument checks of `roi_gather` / `roi_gather_stats` that protect the kernels from output
buffers they would misuse are tested with the library calls replaced by a guard, so that a
missing check fails the test instead of reaching a kernel.
"""
import itertools

import numpy as np
import pytest
import torch

from oracle import reduce as o_red
from oracle import rois as o_rois

pytestmark = pytest.mark.gpu

WARPS = (6, 16, 12, 8, 4)          # the launcher's candidates, in its order of preference
COPY_CLASSES = ("VPL12", "VPL21", "VPL36", "VPL0", "QPL12", "QPL24", "HALF", "GENERIC", "NONE")
FG_CAP, BG_CAP = 1024, 2560        # list capacities: 32 fg and 80 bg values per lane
HIST_WORDS = 256 + 32              # per-warp median histogram


def dev(a, device):
    return torch.from_numpy(np.ascontiguousarray(a)).to(device)


def dev_image(image, device):
    """Device copy of a (C,T,H,W) uint16 image in the layout the staged kernels take: rows
    padded to whole 16-byte vectors (`ops.alloc_image`; dense when W is a multiple of 8)."""
    from magnify_b200 import ops

    out = ops.alloc_image(image.shape, torch.uint16, device)
    out.copy_(dev(image, device))
    return out


# ------------------------------------------------------------------------- launch predictor
def device_limits(device=0):
    """(shared memory per block with opt-in, shared memory per SM, SMs) of the device."""
    p = torch.cuda.get_device_properties(device)
    return p.shared_memory_per_block_optin, p.shared_memory_per_multiprocessor, p.multi_processor_count


def launch_plan(L, C, T, Tm, M, nf_max, nb_max, layout=None, warps=None, limits=None):
    """The host logic of roi_gather_lists restated: None where the fused kernel does not apply
    (the call then takes the dp2a kernels and a separate median pass), else (layout, warps per
    CTA, stages per warp) with layout 1 = one warp per marker, 0 = one CTA per marker.
    layout / warps: what MGB_GATHER_LAYOUT / MGB_GATHER_WARPS force (None: the launcher's choice).
    Only a 16-byte aligned image with a pitch of whole 16-byte vectors is considered."""
    if nf_max > FG_CAP or nb_max > BG_CAP:
        return None
    wpu = (L + 14) & ~7
    if wpu > 256 or L > 256 or (L - 1) * wpu + L + 8 > 65535:
        return None
    max_smem, sm_smem, sms = limits or device_limits()
    stage = (L * wpu * 2 + 127) & ~127
    list_bytes = 2 * (((max(nf_max, 1) + 255) & ~255) + ((max(nb_max, 1) + 255) & ~255))
    items = C * max(1, T // max(1, Tm))
    wpm = items < 128 and M * Tm >= sms * 12 * 8
    if layout is not None:
        wpm = layout == 1
    for _ in range(2):
        pair = not wpm and items < 128
        for cand in WARPS:
            if (cand != warps) if warps else ((cand == 6 and not pair) or (cand == 16 and not wpm)):
                continue
            fixed = (cand if wpm else 1) * list_bytes + cand * HIST_WORDS * 4 + cand * 4 * 8 + T * 4 + 128
            room = sm_smem // 2 - 1024 if cand == 6 else max_smem
            if room < fixed + 1024:
                continue
            one = cand >= 12 or cand == 6
            n = min(1 if one else 4, (room - fixed - 1024) // (cand * stage))
            if n >= (1 if one else 2):
                return int(wpm), cand, n
        if not wpm:
            return None
        wpm = False   # per-warp lists do not fit: one marker per CTA instead
    return None


def expected_fused(L, C, T, Tm, M, nf_max, nb_max, layout=None, warps=None, limits=None):
    """Whether roi_gather_stats takes its summaries from the fused kernel.  The alignment of the
    crop buffer only selects the copy loop (`copy_class`), never whether the kernel applies."""
    return launch_plan(L, C, T, Tm, M, nf_max, nb_max, layout, warps, limits) is not None


def copy_class(L, roi_align):
    """The crop copy loop the launcher compiles in: roi_align is the largest power of two (up to
    16) dividing the crop buffer's byte address, None for summaries only (no crops stored)."""
    if roi_align is None:
        return "NONE"
    if L % 8 == 0 and L > 8 and roi_align >= 16:
        v = (L * (L // 8) + 31) // 32
        return "VPL12" if v <= 12 else "VPL21" if v <= 21 else "VPL36" if v <= 36 else "VPL0"
    q = (L * L // 4 + 31) // 32
    if L % 2 == 0 and roi_align >= 8 and q <= 24:
        return "QPL12" if q <= 12 else "QPL24"
    if L % 2 == 0 and L > 2 and roi_align >= 4:
        return "HALF"
    return "GENERIC"   # (rows of one vector or one word have no division magic number: L = 8, 2 avoid those loops)


def _roi_align(off):
    """Byte alignment of a uint16 crop buffer `off` elements into a fresh allocation."""
    return None if off is None else 16 if off == 0 else min(16, 2 * (off & -off))


# ----------------------------------------------------------------------------- shared helpers
MASK_T = {   # mask timesteps of T = 4 timepoints: Tm and mask_t
    "one": (1, [0, 0, 0, 0]),
    "all": (4, [0, 1, 2, 3]),
    "gap": (3, [0, 0, 2, 2]),        # mask timestep 1 owns no timepoint
    "unsorted": (2, [1, 0, 1, 0]),
}


def _set_env(monkeypatch, layout=None, warps=None):
    for name, value in (("MGB_GATHER_LAYOUT", layout), ("MGB_GATHER_WARPS", warps)):
        if value is None:
            monkeypatch.delenv(name, raising=False)
        else:
            monkeypatch.setenv(name, str(value))
    monkeypatch.delenv("MGB_GATHER_SPLIT", raising=False)


def _exact_masks(rng, length, counts_f, counts_b):
    """Disjoint fg / bg masks with exactly counts_f[i] / counts_b[i] pixels at random positions
    (counts of any shape S -> masks S + (L, L) bool)."""
    counts_f, counts_b = np.asarray(counts_f), np.asarray(counts_b)
    fg = np.zeros(counts_f.shape + (length * length,), dtype=bool)
    bg = np.zeros_like(fg)
    for idx in np.ndindex(counts_f.shape):
        perm = rng.permutation(length * length)
        fg[idx + (perm[:counts_f[idx]],)] = True
        bg[idx + (perm[counts_f[idx]:counts_f[idx] + counts_b[idx]],)] = True
    shape = counts_f.shape + (length, length)
    return fg.reshape(shape), bg.reshape(shape)


def _mask_bytes(rng, mask):
    """uint8 mask with random non-zero bytes where set (the kernels take any non-zero byte)."""
    return (mask * rng.integers(1, 256, mask.shape)).astype(np.uint8)


def _counts(fg, bg):
    return int(fg.sum((-1, -2)).max(initial=0)), int(bg.sum((-1, -2)).max(initial=0))


def _check_stats(got, want, medians=True, msg=""):
    np.testing.assert_array_equal(got[..., :4], want[..., :4], err_msg=msg)
    np.testing.assert_allclose(got[..., 4:6], want[..., 4:6], rtol=1e-12, equal_nan=True, err_msg=msg)
    if medians:
        np.testing.assert_array_equal(got[..., 6:], want[..., 6:], err_msg=msg)
    else:
        assert np.isnan(got[..., 6:]).all(), msg


def _grid_markers(length, m, t, gap=9):
    """Centres of m markers whose windows do not overlap (rows of 8, left edges shifted by
    0..7 pixels so every alignment of the staged window occurs); returns x, y (m, t), image h, w."""
    left = np.array([(i % 8) * (length + gap) + i % 8 for i in range(m)])
    top = np.array([(i // 8) * (length + 3) + 1 for i in range(m)])
    w = 8 * (length + gap) + 8
    h = ((m + 7) // 8) * (length + 3) + 2
    x = np.repeat((left + length // 2).astype(np.float64)[:, None], t, 1)
    y = np.repeat((top + length // 2).astype(np.float64)[:, None], t, 1)
    return x, y, h, w, top, left


# ---------------------------------------------------------------------- configuration matrix
# (L, crop buffer offset in elements: 0 = own allocation, None = no crops)
COPY_CASES = [
    (24, 0), (48, 0),                    # VPL12
    (56, 0), (72, 0),                    # VPL21
    (80, 0), (96, 0),                    # VPL36
    (104, 0),                            # VPL0: run-time vector loop
    (8, 0), (34, 0), (38, 0),            # QPL12 (L = 8: rows of a single vector)
    (42, 0), (50, 0),                    # QPL24
    (58, 0), (70, 0), (72, 4), (34, 2),  # HALF: too many quads, or crops 8 / 4 but not 16 / 8-byte aligned
    (33, 0), (51, 0), (40, 1),           # GENERIC: odd rows, or crops only 2-byte aligned
    (48, None),                          # summaries only
]
C_M, T_M, M_M = 2, 4, 24


def _matrix_masks_max(length):
    """Largest fg / bg pixel count of a matrix case (marker 0 has exactly these)."""
    return min(length * length // 4, 1000), min(length * length // 2, 2000)


def _matrix():
    # (medians, mask timesteps, marker order), dealt round so that both layouts meet each of them
    variants = list(itertools.product((True, False), MASK_T, (False, True)))
    shapes = [(length, off, layout, None) for (length, off), layout in itertools.product(COPY_CASES, (0, 1))]
    shapes += [((24, 42, 58, 33, 72)[i % 5], 0, layout, warps)
               for i, (layout, warps) in enumerate(itertools.product((0, 1), WARPS))]
    return [shape + variants[(i + i // 2) % len(variants)] for i, shape in enumerate(shapes)]


MATRIX = _matrix()


def _matrix_id(case):
    length, off, layout, warps, medians, tmk, order = case
    return (f"L{length}-{'noroi' if off is None else f'off{off}'}-{'wpm' if layout else 'cta'}"
            f"-w{warps or 'auto'}-{'med' if medians else 'nomed'}-{tmk}-{'perm' if order else 'id'}")


def _matrix_plan(case, limits=None):
    length, off, layout, warps, medians, tmk, order = case
    nf, nb = _matrix_masks_max(length)
    return launch_plan(length, C_M, T_M, MASK_T[tmk][0], M_M, nf, nb, layout, warps, limits)


def test_matrix_covers_every_configuration(cuda_device):
    """Every copy class in both layouts, and every warp count, is predicted to run fused in at
    least one case of the matrix (from the list and the predictor alone)."""
    limits = device_limits(cuda_device)
    fused_pairs, fused_warps = set(), set()
    for case in MATRIX:
        plan = _matrix_plan(case, limits)
        if plan is not None:
            fused_pairs.add((copy_class(case[0], _roi_align(case[1])), plan[0]))
            fused_warps.add(plan[1])
    missing = [(cc, lay) for cc in COPY_CLASSES for lay in (0, 1) if (cc, lay) not in fused_pairs]
    assert not missing, f"no fused case for {missing}"
    assert fused_warps == set(WARPS)
    # the copy classes of the list are the ones they are meant to be
    assert {copy_class(length, _roi_align(off)) for length, off in COPY_CASES} == set(COPY_CLASSES)


def _matrix_data(case, seed):
    length, off, layout, warps, medians, tmk, order = case
    rng = np.random.default_rng(seed)
    tm, mask_t = MASK_T[tmk]
    mask_t = np.array(mask_t, dtype=np.int32)
    h, w = length + int(rng.integers(40, 90)), length + int(rng.integers(60, 160))
    image = rng.integers(0, 65535, (C_M, T_M, h, w), dtype=np.uint16, endpoint=True)
    image[1] = np.clip(rng.normal(900, 30, image[1].shape), 0, 65535).astype(np.uint16)   # many ties
    x = rng.uniform(-5, w + 5, (M_M, T_M))
    y = rng.uniform(-5, h + 5, (M_M, T_M))
    nf, nb = _matrix_masks_max(length)
    cf = rng.integers(0, nf + 1, (M_M, tm))
    cb = rng.integers(0, nb + 1, (M_M, tm))
    cf[0, 0], cb[0, -1] = nf, nb                  # the list capacities of the case
    cf[1], cb[2] = 0, 0                           # empty masks: NaN means and medians
    cf[3, 0], cb[3, 0] = 1, 2
    fg, bg = _exact_masks(rng, length, cf, cb)
    return rng, image, x, y, mask_t, tm, fg, bg


@pytest.mark.parametrize("case", MATRIX, ids=[_matrix_id(c) for c in MATRIX])
def test_fused_gather_configuration(cuda_device, monkeypatch, case):
    from magnify_b200 import ops

    length, off, layout, warps, medians, tmk, order = case
    rng, image, x, y, mask_t, tm, fg, bg = _matrix_data(case, MATRIX.index(case))
    _set_env(monkeypatch, layout, warps)
    want_roi = o_rois.gather_rois(image, x, y, length)
    want = o_red.masked_stats(want_roi, fg[:, mask_t], bg[:, mask_t])
    h, w = image.shape[-2:]
    boxes = ops.bounding_boxes(dev(x, cuda_device), dev(y, cuda_device), length, w, h)
    fg_d, bg_d = dev(_mask_bytes(rng, fg), cuda_device), dev(_mask_bytes(rng, bg), cuda_device)
    counts = _counts(fg, bg)
    assert counts == _matrix_masks_max(length)
    shape = (M_M, C_M, T_M, length, length)
    out_roi = None
    if off:
        n = int(np.prod(shape))
        out_roi = torch.empty(n + 8, dtype=torch.uint16, device=cuda_device)[off:off + n].view(shape)
        assert out_roi.data_ptr() % 32 == 2 * off
    perm = dev(rng.permutation(M_M).astype(np.int32), cuda_device) if order else None
    kw = dict(mask_t=dev(mask_t, cuda_device), want_roi=off is not None, out_roi=out_roi, order=perm,
              mask_counts=counts)
    args = (dev_image(image, cuda_device), boxes, fg_d, bg_d, length)
    roi, stats = ops.roi_gather_stats(*args, **kw)
    fused = expected_fused(length, C_M, T_M, tm, M_M, *counts, layout, warps, device_limits(cuda_device))
    assert ops.last_gather_fused is fused
    if off is None:
        assert roi is None
    else:
        np.testing.assert_array_equal(roi.cpu().numpy(), want_roi)
    got = stats.cpu().numpy()
    _check_stats(got, want)
    if not medians:
        # the launcher's choice does not depend on the medians; the sums of the build without
        # them equal the ones above
        _, no_med = ops.roi_gather_stats(*args, **dict(kw, medians=False, out_roi=None))
        no_med = no_med.cpu().numpy()
        np.testing.assert_array_equal(no_med[..., :6], got[..., :6])
        assert np.isnan(no_med[..., 6:]).all()


@pytest.mark.parametrize("step", [0, 1], ids=["largest_fused", "next_falls_back"])
def test_fused_gather_largest_window(cuda_device, monkeypatch, step):
    """The largest L whose stages still fit in shared memory runs fused; one more pixel falls
    back to the dp2a kernels and the median pass, with the same results."""
    from magnify_b200 import ops

    limits = device_limits(cuda_device)
    c, t, m = 1, 2, 12
    largest = max(L for L in range(8, 257) if expected_fused(L, c, t, 1, m, 200, 400, limits=limits))
    length = largest + step
    assert expected_fused(length, c, t, 1, m, 200, 400, limits=limits) is (step == 0)
    _set_env(monkeypatch)
    rng = np.random.default_rng(length)
    h, w = length + 30, length + 70
    image = rng.integers(0, 65535, (c, t, h, w), dtype=np.uint16, endpoint=True)
    x = rng.uniform(0, w, (m, t))
    y = rng.uniform(0, h, (m, t))
    cf, cb = rng.integers(0, 201, (m, 1)), rng.integers(0, 401, (m, 1))
    cf[0], cb[0] = 200, 400
    fg, bg = _exact_masks(rng, length, cf, cb)
    boxes = ops.bounding_boxes(dev(x, cuda_device), dev(y, cuda_device), length, w, h)
    roi, stats = ops.roi_gather_stats(dev_image(image, cuda_device), boxes, dev(fg.view(np.uint8), cuda_device),
                                      dev(bg.view(np.uint8), cuda_device), length, mask_counts=(200, 400))
    assert ops.last_gather_fused is (step == 0)
    want_roi = o_rois.gather_rois(image, x, y, length)
    np.testing.assert_array_equal(roi.cpu().numpy(), want_roi)
    _check_stats(stats.cpu().numpy(), o_red.masked_stats(want_roi, np.repeat(fg, t, 1), np.repeat(bg, t, 1)))


@pytest.mark.parametrize("tma", [1, 0], ids=["staged", "plain"])
@pytest.mark.parametrize("length,dtype,off", [(8, np.uint16, 0), (8, np.uint16, 2), (2, np.uint16, 0),
                                              (2, np.uint16, 2), (4, np.float32, 0), (1, np.float32, 0)])
def test_rows_of_one_vector_or_word(cuda_device, monkeypatch, tma, length, dtype, off):
    """Windows whose rows are a single 16-byte vector (8 uint16 / 4 float32 pixels) or a single
    4-byte word (2 uint16 / 1 float32): the copy loops divide by the vectors / words per row with
    a multiply-high magic number, which does not exist for a divisor of 1, so these rows must take
    other loops.  Crops and summaries on the staged and the plain kernels, crops into a buffer 0 or
    2 elements (16 / 4-byte aligned) into its allocation."""
    from magnify_b200 import _lib, ops

    lib = _lib.load()
    c, t, m = 2, 2, 37
    rng = np.random.default_rng(length * 10 + off)
    h, w = 50, 64
    if dtype == np.uint16:
        image = rng.integers(0, 65535, (c, t, h, w), dtype=np.uint16, endpoint=True)
    else:
        image = rng.random((c, t, h, w)).astype(dtype)
    x = rng.uniform(-3, w + 3, (m, t))
    y = rng.uniform(-3, h + 3, (m, t))
    boxes = ops.bounding_boxes(dev(x, cuda_device), dev(y, cuda_device), length, w, h)
    want_roi = o_rois.gather_rois(image, x, y, length)
    shape = (m, c, t, length, length)
    n = int(np.prod(shape))
    tdtype = torch.uint16 if dtype == np.uint16 else torch.float32
    out = torch.empty(n + 8, dtype=tdtype, device=cuda_device)[off:off + n]
    _set_env(monkeypatch)
    old = lib.mgb_set_tma_enabled(tma)
    try:
        got = ops.roi_gather(dev(image, cuda_device), boxes, length, out=out.view(shape)).cpu().numpy()
        np.testing.assert_array_equal(got, want_roi)
        if dtype != np.uint16:
            return
        fg, bg = _exact_masks(rng, length, rng.integers(0, length * length + 1, (m, 1)), np.zeros((m, 1), int))
        bg = ~fg
        roi, stats = ops.roi_gather_stats(dev(image, cuda_device), boxes, dev(fg.view(np.uint8), cuda_device),
                                          dev(bg.view(np.uint8), cuda_device), length, out_roi=out.view(shape),
                                          mask_counts=_counts(fg, bg))
        assert ops.last_gather_fused is bool(tma)
    finally:
        lib.mgb_set_tma_enabled(old)
    np.testing.assert_array_equal(roi.cpu().numpy(), want_roi)
    _check_stats(stats.cpu().numpy(), o_red.masked_stats(want_roi, np.repeat(fg, t, 1), np.repeat(bg, t, 1)))


# ------------------------------------------------------------- list capacity and padding
def _arranged(kind, n, rng):
    """n pixel values in raster order of a mask; the first (the pixel the list padding repeats)
    is the unique minimum, the unique maximum, the (lower) median, or -- "fine" -- lies in the
    second median pass's window past the coarse bin that holds both middle ranks."""
    if n == 0:
        return np.zeros(0, dtype=np.int64)
    if kind == "min":
        v = rng.integers(1001, 60000, n)
        v[0] = 1000
    elif kind == "max":
        v = rng.integers(20, 300, n)              # range below 256: one-value bins
        v[0] = 300
    elif kind == "median":
        s = np.sort(rng.choice(65536, n, replace=False))
        mid = (n - 1) // 2
        v = np.r_[s[mid], np.delete(s, mid)]
    else:
        # range 2000 -> coarse bins of 8 values; the middle ranks sit on 6000 (bin base 6000),
        # the first pixel on 6100, inside [base + 8, base + 256)
        rest = n - 1
        cluster = min(rest, rest // 3 + 3)
        below = (rest - cluster) // 2
        above = rest - cluster - below
        lows = rng.integers(5000, 5900, below)
        highs = rng.integers(6200, 7001, above)
        if below:
            lows[0] = 5000
        if above:
            highs[0] = 7000
        v = np.r_[6100, lows, np.full(cluster, 6000), highs]
        if n >= 8:
            s = np.sort(v)
            assert s[(n - 1) // 2] == s[n // 2] == 6000 and s[-1] - s[0] == 2000
    head, tail = v[:1], v[1:].copy()
    rng.shuffle(tail)
    v = np.r_[head, tail]
    if kind in ("min", "max") and n > 1:
        assert (v[0] < v[1:]).all() if kind == "min" else (v[0] > v[1:]).all()
    return v


ARRANGEMENTS = ("min", "max", "median", "fine")   # one per (channel, time) window


@pytest.mark.parametrize("which,count", [("fg", n) for n in (0, 1, 2, 255, 256, 257, 1023, 1024, 1025)] +
                         [("bg", n) for n in (2559, 2560, 2561)])
def test_list_capacity_and_padding(cuda_device, monkeypatch, which, count):
    """L = 72: the largest fg (bg) count of the launch sits on, just below or just above a
    multiple of 256 and the capacity of 1024 (2560) pixels, while other markers of the same
    launch have 0 to 3 pixels, so their lists are mostly padding.  The padded pixel is the
    unique minimum, maximum, the median, or in the fine median window.  At most the capacity:
    fused; above it: the dp2a kernels and the median pass, with the same results."""
    from magnify_b200 import ops

    length, c, t, m = 72, 2, 2, 7
    rng = np.random.default_rng(count + (0 if which == "fg" else 7))
    x, y, h, w, top, left = _grid_markers(length, m, t)
    small = np.array([count, 1, 2, 3, 0, 100, count])
    other = np.array([600 if which == "fg" else 300, 1, 2, 3, 0, 50, 40])
    big = np.minimum(small, count)
    cf, cb = (big, other) if which == "fg" else (other, big)
    fg, bg = _exact_masks(rng, length, cf[:, None], cb[:, None])
    image = rng.integers(0, 65535, (c, t, h, w), dtype=np.uint16, endpoint=True)
    for i in range(m):
        for k, (ci, ti) in enumerate(itertools.product(range(c), range(t))):
            win = image[ci, ti, top[i]:top[i] + length, left[i]:left[i] + length]
            for mask in (fg[i, 0], bg[i, 0]):
                win[mask] = _arranged(ARRANGEMENTS[k], int(mask.sum()), rng)
    counts = _counts(fg, bg)
    assert counts[0 if which == "fg" else 1] == count
    fused = count <= (FG_CAP if which == "fg" else BG_CAP)
    assert expected_fused(length, c, t, 1, m, *counts, limits=device_limits(cuda_device)) is fused
    want_roi = o_rois.gather_rois(image, x, y, length)
    want = o_red.masked_stats(want_roi, np.repeat(fg, t, 1), np.repeat(bg, t, 1))
    boxes = ops.bounding_boxes(dev(x, cuda_device), dev(y, cuda_device), length, w, h)
    fg_d, bg_d = dev(fg.view(np.uint8), cuda_device), dev(bg.view(np.uint8), cuda_device)
    for layout in (0, 1):
        _set_env(monkeypatch, layout)
        roi, stats = ops.roi_gather_stats(dev_image(image, cuda_device), boxes, fg_d, bg_d, length, mask_counts=counts)
        assert ops.last_gather_fused is fused
        np.testing.assert_array_equal(roi.cpu().numpy(), want_roi)
        _check_stats(stats.cpu().numpy(), want, msg=f"layout {layout}")


# ------------------------------------------------------------------------- median radix edges
RADIX_KINDS = ("range0", "range1", "range255", "range256", "range257", "range65535", "same_bin", "adjacent_bins",
               "far_apart", "one_high", "one_low", "saturated")


def _radix_values(kind, n, rng):
    """n values whose median exercises one edge of the radix selection (256 bins of the range)."""
    if kind.startswith("range"):
        span = int(kind[5:])
        lo = 0 if span == 65535 else 1200
        v = rng.integers(lo, lo + span + 1, n)
        v[0], v[-1] = lo, lo + span
    elif kind == "same_bin":                      # range 40000: bins of 256; both middles in 20001..20003
        cluster = n // 3 + 3
        below = (n - cluster) // 2
        v = np.r_[rng.integers(0, 19000, below), rng.integers(20001, 20004, cluster),
                  rng.integers(21000, 40001, n - cluster - below)]
        v[0], v[-1] = 0, 40000
    elif kind == "adjacent_bins":                 # middles 20479 | 20480: last value of bin 79, first of bin 80
        half = n // 2
        v = np.r_[rng.integers(0, 20479, half - 1), 20479, 20480, rng.integers(20481, 40001, n - half - 1)]
        v[0], v[-1] = 0, 40000
    elif kind == "far_apart":
        half = n // 2
        v = np.r_[rng.integers(0, 101, half), rng.integers(60000, 65001, n - half)]
    elif kind in ("one_high", "one_low"):
        v = np.full(n, 500)
        v[0] = 9000 if kind == "one_high" else 3
    else:                                         # saturated: 0 and 65535 only
        v = np.where(np.arange(n) < n // 2, 0, 65535)
    rng.shuffle(v)
    return v


@pytest.mark.parametrize("layout", [0, 1], ids=["cta", "wpm"])
def test_median_radix_edges(cuda_device, monkeypatch, layout):
    """Value ranges of 0, 1, 255, 256, 257 and 65535; the two middle ranks in one coarse bin, in
    adjacent bins and far apart; all equal but one; saturated 0 / 65535 -- each with an odd and an
    even pixel count, in the fused medians and in roi_median."""
    from magnify_b200 import ops

    length = 48
    rng = np.random.default_rng(99)
    kinds = [(k, parity) for k in RADIX_KINDS for parity in (1, 0)]
    m, c, t = len(kinds), 1, 1
    x, y, h, w, top, left = _grid_markers(length, m, t)
    cf = np.array([300 + p for _, p in kinds])[:, None]
    cb = np.array([1000 + p for _, p in kinds])[:, None]
    fg, bg = _exact_masks(rng, length, cf, cb)
    image = rng.integers(0, 65535, (c, t, h, w), dtype=np.uint16, endpoint=True)
    for i, (kind, _) in enumerate(kinds):
        win = image[0, 0, top[i]:top[i] + length, left[i]:left[i] + length]
        for mask in (fg[i, 0], bg[i, 0]):
            win[mask] = _radix_values(kind, int(mask.sum()), rng)
    want_roi = o_rois.gather_rois(image, x, y, length)
    want = o_red.masked_stats(want_roi, fg, bg)
    _set_env(monkeypatch, layout)
    boxes = ops.bounding_boxes(dev(x, cuda_device), dev(y, cuda_device), length, w, h)
    fg_d, bg_d = dev(fg.view(np.uint8), cuda_device), dev(bg.view(np.uint8), cuda_device)
    roi, stats = ops.roi_gather_stats(dev_image(image, cuda_device), boxes, fg_d, bg_d, length, mask_counts=_counts(fg, bg))
    assert ops.last_gather_fused is True
    np.testing.assert_array_equal(roi.cpu().numpy(), want_roi)
    _check_stats(stats.cpu().numpy(), want)
    for mask_d, col in ((fg_d, 6), (bg_d, 7)):
        med = ops.roi_median(roi, mask_d).cpu().numpy()
        np.testing.assert_array_equal(med, want[..., col], err_msg=f"roi_median column {col}")


# ------------------------------------------------------------------------------ stale counts
@pytest.mark.parametrize("layout", [0, 1], ids=["cta", "wpm"])
def test_stale_mask_counts_flag_overflowing_markers(cuda_device, monkeypatch, layout):
    """mask_counts below the true counts: a marker whose masks exceed the lists sized from them
    gets exact counts and NaN sums, means and medians -- never a finite wrong number; the other
    markers of the launch are unaffected."""
    from magnify_b200 import ops

    length, c, t, m = 40, 2, 3, 10
    rng = np.random.default_rng(5 + layout)
    h, w = 150, 230
    image = rng.integers(0, 65535, (c, t, h, w), dtype=np.uint16, endpoint=True)
    x = rng.uniform(0, w, (m, t))
    y = rng.uniform(0, h, (m, t))
    cf = rng.integers(0, 251, (m, 1))
    cb = rng.integers(0, 401, (m, 1))
    cf[0], cb[1] = 600, 700                       # over the lists of 512 that (300, 400) give
    fg, bg = _exact_masks(rng, length, cf, cb)
    _set_env(monkeypatch, layout)
    boxes = ops.bounding_boxes(dev(x, cuda_device), dev(y, cuda_device), length, w, h)
    roi, stats = ops.roi_gather_stats(dev_image(image, cuda_device), boxes, dev(fg.view(np.uint8), cuda_device),
                                      dev(bg.view(np.uint8), cuda_device), length, mask_counts=(300, 400))
    assert ops.last_gather_fused is True
    want_roi = o_rois.gather_rois(image, x, y, length)
    want = o_red.masked_stats(want_roi, np.repeat(fg, t, 1), np.repeat(bg, t, 1))
    got = stats.cpu().numpy()
    np.testing.assert_array_equal(roi.cpu().numpy(), want_roi)
    np.testing.assert_array_equal(got[..., :2], want[..., :2])
    assert np.isnan(got[:2, ..., 2:]).all()
    _check_stats(got[2:], want[2:])


# ----------------------------------------------------------------------- pointer alignment
@pytest.mark.parametrize("length", [33, 48])
@pytest.mark.parametrize("offset", [1, 2, 4, 16])
def test_mask_pointer_alignment(cuda_device, monkeypatch, offset, length):
    """fg / bg as contiguous views 1, 2, 4 and 16 bytes into a larger buffer: the byte, 4-byte and
    16-byte mask staging of the fused kernel (with L = 33 every marker's masks start at another
    alignment), in both layouts."""
    from magnify_b200 import ops

    c, t, m = 2, 3, 20
    rng = np.random.default_rng(offset * 100 + length)
    h, w = 140, 210
    image = rng.integers(0, 65535, (c, t, h, w), dtype=np.uint16, endpoint=True)
    x = rng.uniform(0, w, (m, t))
    y = rng.uniform(0, h, (m, t))
    mask_t = np.array([1, 0, 1], dtype=np.int32)
    fg, bg = _exact_masks(rng, length, rng.integers(0, 400, (m, 2)), rng.integers(0, 700, (m, 2)))
    want_roi = o_rois.gather_rois(image, x, y, length)
    want = o_red.masked_stats(want_roi, fg[:, mask_t], bg[:, mask_t])
    boxes = ops.bounding_boxes(dev(x, cuda_device), dev(y, cuda_device), length, w, h)

    def at_offset(mask):
        n = mask.size
        buf = torch.zeros(n + 32, dtype=torch.uint8, device=cuda_device)
        view = buf[offset:offset + n].view(mask.shape)
        view.copy_(dev(_mask_bytes(rng, mask), cuda_device))
        assert view.data_ptr() % 32 == offset
        return view

    fg_d, bg_d = at_offset(fg), at_offset(bg)
    for layout in (0, 1):
        _set_env(monkeypatch, layout)
        roi, stats = ops.roi_gather_stats(dev_image(image, cuda_device), boxes, fg_d, bg_d, length,
                                          mask_t=dev(mask_t, cuda_device), mask_counts=_counts(fg, bg))
        assert ops.last_gather_fused is True
        np.testing.assert_array_equal(roi.cpu().numpy(), want_roi)
        _check_stats(stats.cpu().numpy(), want, msg=f"layout {layout}")


@pytest.mark.parametrize("offset", [1, 4])
def test_dp2a_mask_pointer_alignment(cuda_device, monkeypatch, offset):
    """Masks over the list capacity with many markers and quad rows (L = 34, M = 2048): the
    dp2a kernels read the masks as words only when both are 4-byte aligned (warp-per-marker
    kernel), else byte by byte (CTA kernel); the medians come from the separate pass."""
    from magnify_b200 import ops

    length, c, t, m = 34, 1, 2, 2048
    rng = np.random.default_rng(offset)
    h, w = 300, 700
    image = rng.integers(0, 65535, (c, t, h, w), dtype=np.uint16, endpoint=True)
    x = rng.uniform(0, w, (m, t))
    y = rng.uniform(0, h, (m, t))
    cf = rng.integers(0, 300, (m, 1))
    cf[7] = 1100                                  # over the fg capacity: not fused
    fg, bg = _exact_masks(rng, length, cf, rng.integers(0, 56, (m, 1)))
    want_roi = o_rois.gather_rois(image, x, y, length)
    want = o_red.masked_stats(want_roi, np.repeat(fg, t, 1), np.repeat(bg, t, 1))
    boxes = ops.bounding_boxes(dev(x, cuda_device), dev(y, cuda_device), length, w, h)
    views = []
    for mask in (fg, bg):
        buf = torch.zeros(mask.size + 32, dtype=torch.uint8, device=cuda_device)
        views.append(buf[offset:offset + mask.size].view(mask.shape))
        views[-1].copy_(dev(mask.view(np.uint8), cuda_device))
    _set_env(monkeypatch)
    roi, stats = ops.roi_gather_stats(dev_image(image, cuda_device), boxes, *views, length, mask_counts=_counts(fg, bg))
    assert ops.last_gather_fused is False
    np.testing.assert_array_equal(roi.cpu().numpy(), want_roi)
    _check_stats(stats.cpu().numpy(), want)


@pytest.mark.parametrize("offset", [1, 2])
def test_unaligned_image_takes_plain_kernels(cuda_device, monkeypatch, offset):
    """An image 1 or 2 elements into its buffer cannot be staged (the TMA tensor map needs a
    16-byte aligned base): the plain kernels run, with the median pass, and give the same results."""
    from magnify_b200 import ops

    length, c, t, m = 40, 2, 2, 15
    rng = np.random.default_rng(70 + offset)
    h, w = 120, 200
    image = rng.integers(0, 65535, (c, t, h, w), dtype=np.uint16, endpoint=True)
    buf = torch.zeros(image.size + 16, dtype=torch.uint16, device=cuda_device)
    image_d = buf[offset:offset + image.size].view(image.shape)
    image_d.copy_(dev(image, cuda_device))
    x = rng.uniform(0, w, (m, t))
    y = rng.uniform(0, h, (m, t))
    fg, bg = _exact_masks(rng, length, rng.integers(0, 300, (m, 1)), rng.integers(0, 600, (m, 1)))
    boxes = ops.bounding_boxes(dev(x, cuda_device), dev(y, cuda_device), length, w, h)
    _set_env(monkeypatch)
    roi, stats = ops.roi_gather_stats(image_d, boxes, dev(fg.view(np.uint8), cuda_device),
                                      dev(bg.view(np.uint8), cuda_device), length, mask_counts=_counts(fg, bg))
    assert ops.last_gather_fused is False
    want_roi = o_rois.gather_rois(image, x, y, length)
    np.testing.assert_array_equal(roi.cpu().numpy(), want_roi)
    _check_stats(stats.cpu().numpy(), o_red.masked_stats(want_roi, np.repeat(fg, t, 1), np.repeat(bg, t, 1)))


# ---------------------------------------------------------------------- peer write-out
def _peer_case(rng, device, over_capacity):
    from magnify_b200 import ops

    length, c, t, m = 40, 2, 3, 17
    h, w = 130, 220
    image = rng.integers(0, 65535, (c, t, h, w), dtype=np.uint16, endpoint=True)
    x = rng.uniform(0, w, (m, t))
    y = rng.uniform(0, h, (m, t))
    cf = rng.integers(0, 300, (m, 1))
    if over_capacity:
        cf[4] = 1200
    fg, bg = _exact_masks(rng, length, cf, rng.integers(0, 800, (m, 1)))
    boxes = ops.bounding_boxes(dev(x, device), dev(y, device), length, w, h)
    args = (dev_image(image, device), boxes, dev(fg.view(np.uint8), device), dev(bg.view(np.uint8), device), length)
    want_roi = o_rois.gather_rois(image, x, y, length)
    want = o_red.masked_stats(want_roi, np.repeat(fg, t, 1), np.repeat(bg, t, 1))
    return args, _counts(fg, bg), want_roi, want, (m, c, t, 8)


@pytest.mark.parametrize("path", ["fused", "dp2a"])
@pytest.mark.parametrize("n_peers", [1, 2, 8])
def test_peer_stats_on_one_gpu(cuda_device, monkeypatch, n_peers, path):
    """peer_stats takes plain device addresses, so local buffers stand in for the peers: every
    one of them receives exactly the summaries of the same call without peers (NaN medians on
    the dp2a path, which masks over the list capacity take with medians=False)."""
    from magnify_b200 import ops

    rng = np.random.default_rng(n_peers)
    _set_env(monkeypatch)
    args, counts, want_roi, want, shape = _peer_case(rng, cuda_device, over_capacity=path == "dp2a")
    medians = path == "fused"
    roi, stats = ops.roi_gather_stats(*args, medians=medians, mask_counts=counts)
    local = stats.cpu().numpy()
    _check_stats(local, want, medians=medians)
    bufs = [torch.full(shape, -7.0, dtype=torch.float64, device=cuda_device) for _ in range(n_peers)]
    roi_p, none = ops.roi_gather_stats(*args, medians=medians, mask_counts=counts,
                                       peer_stats=[b.data_ptr() for b in bufs])
    assert none is None
    torch.cuda.synchronize(cuda_device)
    np.testing.assert_array_equal(roi_p.cpu().numpy(), want_roi)
    for j, b in enumerate(bufs):
        np.testing.assert_array_equal(b.cpu().numpy(), local, err_msg=f"peer {j}")


def test_peer_stats_refusals(cuda_device, monkeypatch):
    """Masks over the list capacity cannot give medians through peers (RuntimeError), and more
    than 8 peers are refused by the library before anything is launched."""
    from magnify_b200 import _lib, ops

    rng = np.random.default_rng(3)
    _set_env(monkeypatch)
    args, counts, _, _, shape = _peer_case(rng, cuda_device, over_capacity=True)
    buf = torch.zeros(shape, dtype=torch.float64, device=cuda_device)
    with pytest.raises(RuntimeError, match="peer_stats needs the fused gather"):
        ops.roi_gather_stats(*args, mask_counts=counts, peer_stats=[buf.data_ptr()])
    args, counts, _, _, shape = _peer_case(rng, cuda_device, over_capacity=False)
    bufs = [torch.zeros(shape, dtype=torch.float64, device=cuda_device) for _ in range(9)]
    with pytest.raises(_lib.MagnifyB200Error) as err:
        ops.roi_gather_stats(*args, mask_counts=counts, peer_stats=[b.data_ptr() for b in bufs])
    assert err.value.code == _lib.MGB_EINVAL
    torch.cuda.synchronize(cuda_device)
    assert all(int(torch.count_nonzero(b)) == 0 for b in bufs)


# --------------------------------------------------- output buffers the kernels would misuse
@pytest.fixture
def no_launch(monkeypatch):
    """Replace the library calls by a guard: these tests must be decided by the argument checks."""
    from magnify_b200 import _lib

    def guard(name, *args):
        pytest.fail(f"kernel launched: {name}")

    monkeypatch.setattr(_lib, "call", guard)
    monkeypatch.setattr(_lib, "try_call", guard)


def _small_inputs(device, m=3, c=2, t=2, length=16):
    image = torch.zeros((c, t, 64, 64), dtype=torch.uint16, device=device)
    boxes = torch.zeros((m, t, 2), dtype=torch.int32, device=device)
    fg = torch.ones((m, 1, length, length), dtype=torch.uint8, device=device)
    return image, boxes, fg, fg.clone(), length, (m, c, t, length, length)


def test_roi_gather_rejects_strided_out(cuda_device, no_launch):
    from magnify_b200 import ops

    image, boxes, _, _, length, shape = _small_inputs(cuda_device)
    big = torch.empty(shape[:3] + (length + 2, length + 2), dtype=torch.uint16, device=cuda_device)
    with pytest.raises(ValueError, match="contiguous"):
        ops.roi_gather(image, boxes, length, out=big[..., :length, :length])


def test_roi_gather_stats_rejects_strided_out_roi(cuda_device, no_launch):
    from magnify_b200 import ops

    image, boxes, fg, bg, length, shape = _small_inputs(cuda_device)
    big = torch.empty(shape[:3] + (length, length + 8), dtype=torch.uint16, device=cuda_device)
    with pytest.raises(ValueError, match="contiguous"):
        ops.roi_gather_stats(image, boxes, fg, bg, length, out_roi=big[..., :length], mask_counts=(256, 256))


def test_roi_gather_stats_rejects_misaligned_out_stats(cuda_device, no_launch):
    from magnify_b200 import ops

    image, boxes, fg, bg, length, shape = _small_inputs(cuda_device)
    n = int(np.prod(shape[:3])) * ops.NSTATS
    out = torch.empty(n + 2, dtype=torch.float64, device=cuda_device)[1:n + 1].view(shape[:3] + (ops.NSTATS,))
    assert out.is_contiguous() and out.data_ptr() % 16 == 8
    for medians in (True, False):
        with pytest.raises(ValueError, match="16-byte aligned"):
            ops.roi_gather_stats(image, boxes, fg, bg, length, out_stats=out, medians=medians, mask_counts=(256, 256))


def test_roi_gather_stats_rejects_misaligned_peer_stats(cuda_device, no_launch):
    from magnify_b200 import ops

    image, boxes, fg, bg, length, shape = _small_inputs(cuda_device)
    bufs = [torch.empty(shape[:3] + (ops.NSTATS + 2,), dtype=torch.float64, device=cuda_device) for _ in range(2)]
    for peers in ([bufs[0].data_ptr() + 8], [bufs[0].data_ptr(), bufs[1].data_ptr() + 8]):
        with pytest.raises(ValueError, match="16-byte aligned"):
            ops.roi_gather_stats(image, boxes, fg, bg, length, peer_stats=peers, mask_counts=(256, 256))
