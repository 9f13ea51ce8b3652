"""Parity of the CUDA path (through the C ABI) against the CPU oracle and the golden fixtures.

Integer / byte / index results must be bit-exact; the float summaries must agree to 1e-5
relative (north_star) -- they are in fact exact rationals rounded once, so the test uses 1e-12.
"""
import numpy as np
import pytest
import torch

from oracle import flatfield as o_ff
from oracle import geometry as o_geo
from oracle import reduce as o_red
from oracle import rois as o_rois
from oracle import stitch as o_st

pytestmark = pytest.mark.gpu


def dev(a, device):
    return torch.from_numpy(np.ascontiguousarray(a)).to(device)


@pytest.fixture(params=["staged_cpasync", "staged_tma", "plain"])
def gather_path(request, cuda_device):
    """Run the ROI-gather tests through every implementation: windows staged in shared memory by
    TMA tensor copies (the default) or by cp.async chunks, and the plain load/store kernels."""
    from magnify_b200 import _lib

    lib = _lib.load()
    old_tma = lib.mgb_set_tma_enabled(0 if request.param == "plain" else 1)
    old_loader = lib.mgb_set_gather_loader(0 if request.param == "staged_tma" else 1)
    yield request.param
    lib.mgb_set_tma_enabled(old_tma)
    lib.mgb_set_gather_loader(old_loader)


# ------------------------------------------------------------------------------------ stitch
@pytest.mark.parametrize(
    "shape,overlap,dtype",
    [
        ((1, 1, 2, 3, 40, 40), 5, np.float64),     # reference tests/test_stitch.py:9-26
        ((1, 1, 1, 1, 30, 30), 5, np.float64),     # :28-45
        ((2, 3, 2, 2, 25, 25), 8, np.float64),     # :47-76 (odd pitch -> element-wise kernel)
        ((1, 1, 1, 2, 20, 20), 0, np.float64),     # :78-96
        ((2, 2, 3, 4, 64, 64), 6, np.uint16),      # vector path, phases 0/2/4/6 like 2048/102
        ((1, 2, 2, 5, 48, 56), 7, np.uint16),      # odd overlap, odd phases
        ((1, 1, 2, 2, 32, 40), 9, np.uint8),       # 1-byte elements
        ((2, 1, 2, 3, 32, 32), 4, np.float32),     # 4-byte elements
        ((1, 1, 3, 3, 16, 24), 0, np.uint16),
        ((0, 1, 2, 2, 16, 16), 2, np.uint16),      # empty
    ],
)
def test_stitch_matches_oracle(cuda_device, shape, overlap, dtype):
    from magnify_b200 import ops

    rng = np.random.default_rng(1)
    if np.issubdtype(dtype, np.floating):
        tiles = rng.random(shape).astype(dtype)
    else:
        tiles = rng.integers(0, np.iinfo(dtype).max, shape, dtype=dtype, endpoint=True)
    want = o_st.stitch(tiles, overlap)
    got = ops.stitch(dev(tiles, cuda_device), overlap).cpu().numpy()
    assert got.dtype == want.dtype and got.shape == want.shape
    np.testing.assert_array_equal(got, want)


def test_stitch_reference_golden_slices(cuda_device):
    """The exact-slice assertions of the reference's tests/test_stitch.py:22-26,43-45,93-96."""
    from magnify_b200 import ops

    tile_data = np.random.rand(1, 1, 2, 3, 40, 40)
    img = ops.stitch(dev(tile_data, cuda_device), 5).cpu().numpy()
    assert img.shape[-2:] == (2 * 35, 3 * 35)
    np.testing.assert_array_equal(img[0, 0, 35:70, 35:70], tile_data[0, 0, 1, 1, 2:37, 2:37])
    tile_data = np.random.rand(1, 1, 1, 1, 30, 30)
    img = ops.stitch(dev(tile_data, cuda_device), 5).cpu().numpy()
    np.testing.assert_array_equal(img[0, 0], tile_data[0, 0, 0, 0, 2:27, 2:27])
    tile_data = np.random.rand(1, 1, 1, 2, 20, 20)
    img = ops.stitch(dev(tile_data, cuda_device), 0).cpu().numpy()
    np.testing.assert_array_equal(img[0, 0, :, :20], tile_data[0, 0, 0, 0])
    np.testing.assert_array_equal(img[0, 0, :, 20:], tile_data[0, 0, 0, 1])


def test_stitch_golden_from_reference_source(cuda_device, golden):
    """CUDA stitch against the outputs of the reference's own Stitcher source (tests/golden/stitch.npz)."""
    from magnify_b200 import ops

    g = golden("stitch")
    for name in ("odd", "even", "zero", "single", "max"):
        got = ops.stitch(dev(g[name + "__tiles"], cuda_device), int(g[name + "__overlap"]))
        np.testing.assert_array_equal(got.cpu().numpy(), g[name + "__image"], err_msg=name)


def test_stitch_errors(cuda_device):
    from magnify_b200 import ops

    t = torch.zeros((1, 1, 2, 2, 50, 50), dtype=torch.uint16, device=cuda_device)
    with pytest.raises(ValueError):
        ops.stitch(t, -5)      # tests/test_stitch.py:98-100
    with pytest.raises(ValueError):
        ops.stitch(t, 100)     # tests/test_stitch.py:112-125


# -------------------------------------------------------------------------------- flat-field
def _ff_case(rng, shape, per_channel=False, scalar_dark=False):
    c, t, r, cc, h, w = shape
    tiles = np.clip(rng.normal(3000, 1500, shape), 0, 65535).astype(np.uint16)
    tiles[..., :3, :] = 0          # pixels below dark -> clipped to 0
    tiles[0, 0, 0, 0, 5, 5] = 65535
    yy, xx = np.mgrid[0:h, 0:w]
    flat = 1.0 + 0.35 * np.cos(yy / h * 2.1) * np.sin(xx / w * 1.7 + 0.3)
    dark = 100.0 + 5.0 * np.sin(yy * 0.37 + xx * 0.11)
    if per_channel:
        flat = np.stack([flat * (1 + 0.1 * k) for k in range(c)])[:, None, None, None]
        dark = np.stack([dark + 3 * k for k in range(c)])[:, None, None, None]
    if scalar_dark:
        dark = 97.25
    return tiles, flat, dark


@pytest.mark.parametrize(
    "shape,overlap,per_channel,scalar_dark",
    [
        ((2, 3, 2, 2, 64, 64), 6, False, False),
        ((2, 2, 1, 4, 64, 64), 6, True, False),
        ((1, 2, 2, 3, 48, 56), 7, False, True),
        ((3, 1, 1, 1, 128, 128), 0, True, True),
        ((1, 2, 2, 2, 50, 50), 4, False, False),   # W % 8 != 0 -> generic exact path + stitch
    ],
)
def test_flatfield_stitch_bit_exact(cuda_device, shape, overlap, per_channel, scalar_dark):
    from magnify_b200 import ops

    rng = np.random.default_rng(3)
    tiles, flat, dark = _ff_case(rng, shape, per_channel, scalar_dark)
    want_tiles = o_ff.flatfield_correct(tiles, flat, dark)
    want = o_st.stitch(want_tiles, overlap)
    plan = ops.FlatFieldPlan(shape, flat, dark, device=cuda_device)
    got = ops.flatfield_stitch(dev(tiles, cuda_device), overlap=overlap, plan=plan)
    m_want = o_ff.flatfield_maxima(tiles, flat, dark)
    assert tuple(plan.maxima.cpu().numpy()) == m_want           # bit-exact float64 maxima
    np.testing.assert_array_equal(got.cpu().numpy(), want)
    got_tiles = ops.flatfield_correct(dev(tiles, cuda_device), flat, dark)
    np.testing.assert_array_equal(got_tiles.cpu().numpy(), want_tiles)


def test_flatfield_degenerate_coefficients_take_exact_path(cuda_device):
    """flat = 1, integer dark: every corrected value is an exact integer, so every pixel sits on
    the guard band and must come out of the exact path."""
    from magnify_b200 import ops

    rng = np.random.default_rng(5)
    shape = (1, 2, 2, 2, 32, 32)
    tiles = rng.integers(0, 65535, shape, dtype=np.uint16, endpoint=True)
    for flat, dark in [(1.0, 100.0), (np.ones((32, 32)), np.full((32, 32), 7.0)), (0.5, 0.0), (2.0, 1.5)]:
        want = o_st.stitch(o_ff.flatfield_correct(tiles, flat, dark), 4)
        got = ops.flatfield_stitch(dev(tiles, cuda_device), flat, dark, overlap=4)
        np.testing.assert_array_equal(got.cpu().numpy(), want)
    # the defaults are the identity (preprocess.py:62 with registry.py:278-279)
    got = ops.flatfield_stitch(dev(tiles, cuda_device), 1.0, 0.0, overlap=4)
    np.testing.assert_array_equal(got.cpu().numpy(), o_st.stitch(o_ff.flatfield_correct(tiles), 4))


@pytest.mark.parametrize("dtype", [np.float32, np.float64, np.uint8])
def test_flatfield_other_dtypes(cuda_device, dtype):
    from magnify_b200 import ops

    rng = np.random.default_rng(6)
    shape = (2, 1, 2, 2, 24, 32)
    if dtype == np.uint8:
        tiles = rng.integers(0, 255, shape, dtype=np.uint8, endpoint=True)
        dark = 3.5
    else:
        tiles = (rng.random(shape) * 4000).astype(dtype)
        dark = 100.25
    flat = 0.7 + 0.6 * rng.random((24, 32))
    want = o_st.stitch(o_ff.flatfield_correct(tiles, flat, dark), 2)
    got = ops.flatfield_stitch(dev(tiles, cuda_device), flat, dark, overlap=2)
    np.testing.assert_array_equal(got.cpu().numpy(), want)


def test_flatfield_golden_from_reference_source(cuda_device, golden):
    """CUDA path against the outputs of the reference's own flatfield_correct source
    (tests/golden/flatfield.npz, made by tests/golden/make_golden.py::golden_flatfield)."""
    from magnify_b200 import ops

    g = golden("flatfield")
    tiles = dev(g["tiles"], cuda_device)
    for name in ("arrays", "scalars", "defaults", "integer_dark", "per_channel", "scalar_flat_array_dark"):
        f, d = g[name + "__flat"], g[name + "__dark"]
        f = float(f) if f.ndim == 0 else f
        d = float(d) if d.ndim == 0 else d
        got = ops.flatfield_correct(tiles, f, d)
        np.testing.assert_array_equal(got.cpu().numpy(), g[name + "__out"], err_msg=name)
    got = ops.flatfield_correct(dev(g["f32_tiles"], cuda_device), g["arrays__flat"][:16, :24], g["arrays__dark"][:16, :24])
    np.testing.assert_array_equal(got.cpu().numpy(), g["f32__out"])


def test_flatfield_rejects_nonpositive_flat(cuda_device):
    from magnify_b200 import ops

    with pytest.raises(ValueError):
        ops.FlatFieldPlan((1, 1, 1, 1, 8, 8), np.zeros((8, 8)), 0.0, device=cuda_device)


# ------------------------------------------------------------------------------------- boxes
def test_bounding_boxes_golden(cuda_device, golden):
    from magnify_b200 import ops

    g = golden("geometry")
    args, out = g["bb_args"], g["bb_out"]
    ok = (args[:, 3] >= args[:, 2]) & (args[:, 4] >= args[:, 2])   # image at least as large as the box
    for length in np.unique(args[ok, 2])[:40]:
        for (w, h) in {(int(a[3]), int(a[4])) for a in args[ok & (args[:, 2] == length)]}:
            sel = ok & (args[:, 2] == length) & (args[:, 3] == w) & (args[:, 4] == h)
            x = dev(args[sel, 0].astype(np.float64), cuda_device)
            y = dev(args[sel, 1].astype(np.float64), cuda_device)
            boxes = ops.bounding_boxes(x, y, int(length), w, h).cpu().numpy()
            np.testing.assert_array_equal(boxes[:, 0], out[sel, 0])
            np.testing.assert_array_equal(boxes[:, 1], out[sel, 2])


def test_bounding_boxes_round_half_even(cuda_device):
    from magnify_b200 import ops

    xs = np.array([0.5, 1.5, 2.5, 3.5, 10.49999, 10.5, 11.5, 99.5, 100.5, -0.5, 250.5, 251.5])
    ys = xs[::-1].copy()
    boxes, rel = ops.bounding_boxes(dev(xs, cuda_device), dev(ys, cuda_device), 21, 300, 280, want_rel=True)
    want = o_geo.boxes_from_centres(xs, ys, 21, 300, 280)
    np.testing.assert_array_equal(boxes.cpu().numpy(), want)
    for i in range(len(xs)):
        assert rel[i, 0].item() == round(float(ys[i])) - want[i, 0]
        assert rel[i, 1].item() == round(float(xs[i])) - want[i, 1]


# ------------------------------------------------------------------------------- beads golden
def test_beads_golden(cuda_device, golden, make_pattern_image, gather_path):
    """Labels, fg/bg and ROI crops of BeadFinder's ROI half (find.py:561-602) -- fixture made
    with the reference's real utils.py."""
    from magnify_b200 import ops

    g = golden("beads")
    c, t, h, w = (int(v) for v in g["image_shape"])
    length = int(g["roi_length"])
    image = make_pattern_image(c, t, h, w, salt=int(g["image_salt"]))
    beads = g["beads"]
    m = len(beads)
    beads_i = dev(beads.astype(np.int32), cuda_device)
    labels = ops.bead_labels(beads_i, h, w)
    np.testing.assert_array_equal(labels.cpu().numpy(), g["labels"])
    # beads handed over from the host (the component path: no device read of the radius range)
    labels_h = ops.bead_labels(beads.astype(np.int32), h, w, device=cuda_device)
    np.testing.assert_array_equal(labels_h.cpu().numpy(), g["labels"])
    with pytest.raises(ValueError):
        ops.bead_labels(np.array([[5, 5, 0]], dtype=np.int32), h, w, device=cuda_device)
    x = dev(np.repeat(beads[:, 1:2], t, axis=1), cuda_device)
    y = dev(np.repeat(beads[:, 0:1], t, axis=1), cuda_device)
    boxes = ops.bounding_boxes(x, y, length, w, h)
    np.testing.assert_array_equal(boxes[:, 0].cpu().numpy(), g["boxes"][:, [0, 2]])
    fg, bg, counts = ops.bead_masks(labels, boxes[:, 0].contiguous(), length, want_counts=True)
    np.testing.assert_array_equal(fg.cpu().numpy().astype(bool), g["fg"])
    np.testing.assert_array_equal(bg.cpu().numpy().astype(bool), g["bg"])
    np.testing.assert_array_equal(counts.cpu().numpy(), np.stack([g["fg"].sum((1, 2)), g["bg"].sum((1, 2))], 1))
    roi, stats = ops.roi_gather_stats(dev(image, cuda_device), boxes, fg[:, None].contiguous(),
                                      bg[:, None].contiguous(), length)
    np.testing.assert_array_equal(roi.cpu().numpy(), g["roi"])
    roi2 = ops.roi_gather(dev(image, cuda_device), boxes, length)
    np.testing.assert_array_equal(roi2.cpu().numpy(), g["roi"])
    want = o_red.masked_stats(g["roi"], np.repeat(g["fg"][:, None], t, 1), np.repeat(g["bg"][:, None], t, 1))
    np.testing.assert_allclose(stats.cpu().numpy(), want, rtol=1e-12, equal_nan=True)
    for mask, key in ((fg, "fg"), (bg, "bg")):
        med = ops.roi_median(roi, mask[:, None].contiguous())
        want_med = o_red.masked_median(g["roi"], np.repeat(g[key][:, None], t, 1))
        np.testing.assert_array_equal(med.cpu().numpy(), want_med)
    assert m == roi.shape[0]


def test_beads_zero_markers(cuda_device, gather_path):
    """find.py:557-558 / tests/test_beads.py:219-232: no beads -> empty mark dimension."""
    from magnify_b200 import ops

    image = torch.zeros((2, 1, 64, 64), dtype=torch.uint16, device=cuda_device)
    beads = torch.zeros((0, 3), dtype=torch.int32, device=cuda_device)
    labels = ops.bead_labels(beads, 64, 64)
    assert int((labels != -1).sum()) == 0
    boxes = torch.zeros((0, 1, 2), dtype=torch.int32, device=cuda_device)
    roi = ops.roi_gather(image, boxes, 20)
    assert tuple(roi.shape) == (0, 2, 1, 20, 20)
    fg, bg = ops.bead_masks(labels, boxes[:, 0].contiguous(), 20)
    roi, stats = ops.roi_gather_stats(image, boxes, fg[:, None].contiguous(), bg[:, None].contiguous(), 20)
    assert tuple(stats.shape) == (0, 2, 1, 8)


# -------------------------------------------------------------------------------- chip golden
def test_chip_golden(cuda_device, golden, make_pattern_image, gather_path):
    """ROI crops + disc/annulus masks of ButtonFinder.find_rois and the copy-forward loop
    (find.py:143-176, 362-400) -- fixture made with the reference's real utils.py (cv.circle)."""
    from magnify_b200 import ops

    g = golden("chip")
    c, t, h, w = (int(v) for v in g["image_shape"])
    length = int(g["roi_length"])
    image = make_pattern_image(c, t, h, w, salt=int(g["image_salt"]))
    x = g["x"].reshape(-1)
    y = g["y"].reshape(-1)
    m = len(x)
    xt = dev(np.repeat(x[:, None], t, 1), cuda_device)
    yt = dev(np.repeat(y[:, None], t, 1), cuda_device)
    boxes, rel = ops.bounding_boxes(xt, yt, length, w, h, want_rel=True)
    fg, bg = ops.chip_masks(rel[:, 0].contiguous(), dev(g["fg_radius"].reshape(-1).astype(np.int32), cuda_device),
                            int(g["max_button_radius"]), int(g["chamber_radius"]), length)
    np.testing.assert_array_equal(fg.cpu().numpy().astype(bool), g["fg"][:, 0])
    np.testing.assert_array_equal(bg.cpu().numpy().astype(bool), g["bg"][:, 0])
    roi, stats = ops.roi_gather_stats(dev(image, cuda_device), boxes, fg[:, None].contiguous(),
                                      bg[:, None].contiguous(), length)
    np.testing.assert_array_equal(roi.cpu().numpy(), g["roi"])
    want = o_red.masked_stats(g["roi"], g["fg"], g["bg"])
    np.testing.assert_allclose(stats.cpu().numpy(), want, rtol=1e-12, equal_nan=True)
    med = ops.roi_median(roi, bg[:, None].contiguous())
    np.testing.assert_array_equal(med.cpu().numpy(), o_red.masked_median(g["roi"], g["bg"]))
    assert m == 6


def test_chip_masks_cv_golden(cuda_device, golden):
    from magnify_b200 import ops

    g = golden("masks_cv")
    cases = g["cases"]
    for (ro, ri) in {(int(a[3]), int(a[4])) for a in cases}:
        sel = (cases[:, 3] == ro) & (cases[:, 4] == ri)
        rel = dev(cases[sel][:, :2].astype(np.int32), cuda_device)
        rad = dev(cases[sel][:, 2].astype(np.int32), cuda_device)
        fg, bg, counts = ops.chip_masks(rel, rad, ri, ro, 72, want_counts=True)
        np.testing.assert_array_equal(fg.cpu().numpy().astype(bool), g["disc"][sel])
        np.testing.assert_array_equal(bg.cpu().numpy().astype(bool), g["ring"][sel])
        np.testing.assert_array_equal(counts[:, 0].cpu().numpy(), g["disc"][sel].sum((1, 2)))


# --------------------------------------------------------------------- randomized vs oracle
@pytest.mark.parametrize("length,itemsize_dtype", [(72, np.uint16), (50, np.uint16), (51, np.uint16), (100, np.uint16),
                                                    (24, np.float32), (17, np.uint8), (16, np.float64)])
def test_roi_gather_random(cuda_device, length, itemsize_dtype, gather_path):
    from magnify_b200 import ops

    rng = np.random.default_rng(11)
    c, t, h, w, m = 3, 2, 260, 333 if length % 2 else 336, 37
    if np.issubdtype(itemsize_dtype, np.floating):
        image = rng.random((c, t, h, w)).astype(itemsize_dtype)
    else:
        image = rng.integers(0, np.iinfo(itemsize_dtype).max, (c, t, h, w), dtype=itemsize_dtype, endpoint=True)
    x = rng.uniform(-20, w + 20, (m, t))
    y = rng.uniform(-20, h + 20, (m, t))
    x[:4] = np.round(x[:4]) + 0.5          # exact ties
    want = o_rois.gather_rois(image, x, y, length)
    boxes = ops.bounding_boxes(dev(x, cuda_device), dev(y, cuda_device), length, w, h)
    got = ops.roi_gather(dev(image, cuda_device), boxes, length)
    np.testing.assert_array_equal(got.cpu().numpy(), want)


def test_median_random(cuda_device):
    from magnify_b200 import ops

    rng = np.random.default_rng(12)
    for length in (8, 50, 72, 100, 128):
        m, c, t = 9, 2, 2
        roi = rng.integers(390, 420, (m, c, t, length, length)).astype(np.uint16)   # many ties
        roi[0] = rng.integers(0, 65535, roi[0].shape, endpoint=True)
        mask = rng.random((m, t, length, length)) < 0.3
        mask[1] = False                       # empty -> NaN
        mask[2, :, 0, :3] = True
        mask[3] = True
        got = ops.roi_median(dev(roi, cuda_device), dev(mask.view(np.uint8), cuda_device)).cpu().numpy()
        want = o_red.masked_median(roi, mask)
        np.testing.assert_array_equal(got, want)


def test_full_size_properties_c2(cuda_device, gather_path):
    """BASELINE config 2 at full size (4x4 tiles of 2048^2, overlap 102, 56x32 buttons, L=72):
    size-independent properties instead of a CPU replay -- the stitched image equals torch
    indexing of the tiles, ROI crops equal direct slices, sums of masked sums match."""
    from magnify_b200 import ops

    torch.manual_seed(0)
    c, t, r, cc, h, w, ov, length = 2, 1, 4, 4, 2048, 2048, 102, 72
    tiles = torch.randint(0, 65536, (c, t, r, cc, h, w), dtype=torch.int32, device=cuda_device).to(torch.uint16)
    image = ops.stitch(tiles, ov)
    kept = tiles[..., 51:2048 - 51, 51:2048 - 51]
    ref = kept.permute(0, 1, 2, 4, 3, 5).reshape(c, t, r * 1946, cc * 1946)
    assert torch.equal(image.view(torch.int16), ref.contiguous().view(torch.int16))
    rows, cols = 56, 32
    gy, gx = torch.meshgrid(torch.arange(rows, dtype=torch.float64), torch.arange(cols, dtype=torch.float64), indexing="ij")
    x = (300.25 + gx * 232.9).reshape(-1, 1).to(cuda_device).contiguous()
    y = (350.5 + gy * 126.1).reshape(-1, 1).to(cuda_device).contiguous()
    boxes, rel = ops.bounding_boxes(x, y, length, image.shape[-1], image.shape[-2], want_rel=True)
    rad = torch.full((rows * cols,), 15, dtype=torch.int32, device=cuda_device)
    fg, bg = ops.chip_masks(rel[:, 0].contiguous(), rad, 15, 30, length)
    roi, stats = ops.roi_gather_stats(image, boxes, fg[:, None].contiguous(), bg[:, None].contiguous(), length)
    for m in (0, 17, 1000, rows * cols - 1):
        top, left = (int(v) for v in boxes[m, 0])
        assert torch.equal(roi[m, :, 0].contiguous().view(torch.int16),
                           image[:, 0, top:top + length, left:left + length].contiguous().view(torch.int16))
    sums = (roi.to(torch.float64) * fg[:, None, None].to(torch.float64)).sum((-1, -2))
    assert torch.equal(sums, stats[..., 2])
    assert torch.equal(stats[..., 0], fg.sum((-1, -2)).to(torch.float64)[:, None, None].expand(-1, c, t))


@pytest.mark.parametrize("length", [72, 50, 33])
def test_gather_stats_random_masks(cuda_device, gather_path, length):
    """Fused gather + masked sums with arbitrary (overlapping, empty, full) masks and several
    mask timesteps (chip with more than one search timestep, find.py:151,172-173)."""
    from magnify_b200 import ops

    rng = np.random.default_rng(21)
    c, t, h, w, m = 3, 5, 200, 256, 11
    image = rng.integers(0, 65535, (c, t, h, w), dtype=np.uint16, endpoint=True)
    x = rng.uniform(0, w, (m, t))
    y = rng.uniform(0, h, (m, t))
    mask_t = np.array([0, 0, 1, 1, 1], dtype=np.int32)
    fg = rng.random((m, 2, length, length)) < 0.3
    bg = rng.random((m, 2, length, length)) < 0.5
    fg[0] = False
    bg[1] = True
    want_roi = o_rois.gather_rois(image, x, y, length)
    want = o_red.masked_stats(want_roi, fg[:, mask_t], bg[:, mask_t])
    boxes = ops.bounding_boxes(dev(x, cuda_device), dev(y, cuda_device), length, w, h)
    roi, stats = ops.roi_gather_stats(dev(image, cuda_device), boxes, dev(fg.view(np.uint8), cuda_device),
                                      dev(bg.view(np.uint8), cuda_device), length, mask_t=dev(mask_t, cuda_device))
    np.testing.assert_array_equal(roi.cpu().numpy(), want_roi)
    np.testing.assert_allclose(stats.cpu().numpy(), want, rtol=1e-12, equal_nan=True)
    _, stats2 = ops.roi_gather_stats(dev(image, cuda_device), boxes, dev(fg.view(np.uint8), cuda_device),
                                     dev(bg.view(np.uint8), cuda_device), length, mask_t=dev(mask_t, cuda_device),
                                     want_roi=False)
    np.testing.assert_allclose(stats2.cpu().numpy(), want, rtol=1e-12, equal_nan=True)


def test_flatfield_extreme_coefficients(cuda_device):
    """Flat fields with a huge dynamic range.  (a) wild values everywhere; (b) a dim band with a
    tiny flat value next to bright pixels with flat = 1: there gain = (1/f)(M/M2) exceeds the fast
    path's budget (gain > 16), the positions are encoded as "always exact" (gain 0) and must still
    be bit-exact, mixed with ordinary positions in the same 8-pixel vectors."""
    from magnify_b200 import ops

    rng = np.random.default_rng(31)
    shape = (2, 3, 2, 2, 64, 64)
    tiles = rng.integers(0, 65535, shape, dtype=np.uint16, endpoint=True)
    flat = np.exp(rng.uniform(np.log(0.004), np.log(3.0), (64, 64)))
    flat[::7, ::5] = 1e-6
    flat[3, :] = 1e3
    dark = rng.uniform(0, 300, (64, 64))
    dark[:, ::9] = 0.0
    want = o_st.stitch(o_ff.flatfield_correct(tiles, flat, dark), 6)
    plan = ops.FlatFieldPlan(shape, flat, dark, device=cuda_device)
    got = ops.flatfield_stitch(dev(tiles, cuda_device), overlap=6, plan=plan)
    assert tuple(plan.maxima.cpu().numpy()) == o_ff.flatfield_maxima(tiles, flat, dark)
    np.testing.assert_array_equal(got.cpu().numpy(), want)

    tiles_b = tiles.copy()
    tiles_b[..., 10:20, :] = rng.integers(100, 400, tiles_b[..., 10:20, :].shape)
    flat_b = np.ones((64, 64))
    flat_b[10:20, 3::4] = 0.01
    dark_b = np.full((64, 64), 100.0)
    want = o_st.stitch(o_ff.flatfield_correct(tiles_b, flat_b, dark_b), 6)
    plan = ops.FlatFieldPlan(shape, flat_b, dark_b, device=cuda_device)
    got = ops.flatfield_stitch(dev(tiles_b, cuda_device), overlap=6, plan=plan)
    np.testing.assert_array_equal(got.cpu().numpy(), want)
    gain = plan.gain.cpu().numpy()
    assert (gain[0, 10:20, 3::4] == 0).all() and (gain[0, 30:, :] > 0).all()   # both encodings exercised


@pytest.mark.parametrize("length", [50, 34, 22])
def test_gather_warp_per_marker_kernel(cuda_device, length):
    """Many markers x few windows (bead-screen shape) takes the warp-per-marker quad kernel: it
    must agree bit for bit with the CTA-per-marker staged kernel and the plain kernels, and with
    the oracle on a sample of markers."""
    from magnify_b200 import _lib, ops

    lib = _lib.load()
    rng = np.random.default_rng(41)
    c, t, h, w, m = 2, 3, 600, 1024, 3000
    image = rng.integers(0, 65535, (c, t, h, w), dtype=np.uint16, endpoint=True)
    x = rng.uniform(-10, w + 10, (m, t))
    y = rng.uniform(-10, h + 10, (m, t))
    mask_t = np.array([0, 1, 1], dtype=np.int32)
    fg = rng.random((m, 2, length, length)) < 0.25
    bg = rng.random((m, 2, length, length)) < 0.5
    fg[5] = False
    image_d = dev(image, cuda_device)
    boxes = ops.bounding_boxes(dev(x, cuda_device), dev(y, cuda_device), length, w, h)
    args = (image_d, boxes, dev(fg.view(np.uint8), cuda_device), dev(bg.view(np.uint8), cuda_device), length)
    order = ops.spatial_order(boxes)
    results = {}
    for name, tma, loader in (("wpm", 1, 0), ("cta", 1, 2), ("plain", 0, 0)):
        old_t, old_l = lib.mgb_set_tma_enabled(tma), lib.mgb_set_gather_loader(loader)
        try:
            roi, stats = ops.roi_gather_stats(*args, mask_t=dev(mask_t, cuda_device), order=order if name == "wpm" else None)
            _, stats_only = ops.roi_gather_stats(*args, mask_t=dev(mask_t, cuda_device), want_roi=False)
            roi_only = ops.roi_gather(image_d, boxes, length)
        finally:
            lib.mgb_set_tma_enabled(old_t)
            lib.mgb_set_gather_loader(old_l)
        results[name] = (roi.cpu().numpy(), stats.cpu().numpy(), stats_only.cpu().numpy(), roi_only.cpu().numpy())
    for name in ("cta", "plain"):
        for a, b in zip(results["wpm"], results[name]):
            np.testing.assert_array_equal(a, b, err_msg=name)
    sample = np.r_[0:8, 1500:1504, m - 4:m]
    want_roi = o_rois.gather_rois(image, x[sample], y[sample], length)
    np.testing.assert_array_equal(results["wpm"][0][sample], want_roi)
    want = o_red.masked_stats(want_roi, fg[sample][:, mask_t], bg[sample][:, mask_t])
    np.testing.assert_allclose(results["wpm"][1][sample], want, rtol=1e-12, equal_nan=True)


# ------------------------------------------------------------------- padded image rows
@pytest.mark.parametrize("shape,overlap", [((2, 2, 3, 3, 64, 64), 6), ((1, 2, 2, 5, 64, 72), 7), ((1, 1, 3, 3, 2048, 2048), 102)])
def test_unaligned_image_width_uses_padded_rows(cuda_device, shape, overlap, gather_path):
    """Tile grids whose stitched width is not a multiple of 8 pixels (3x3, 5x5, 10x10 at overlap
    102 ...): the image is allocated with a padded row pitch so the vectorised stitch, the fused
    flat-field kernel and the staged gather still apply; values equal the oracle's dense arrays."""
    from magnify_b200 import ops

    rng = np.random.default_rng(50)
    c, t, r, cc, h, w = shape
    wim, him = cc * (w - overlap), r * (h - overlap)
    assert wim % 8 != 0
    tiles = rng.integers(0, 65535, shape, dtype=np.uint16, endpoint=True)
    tiles_d = dev(tiles, cuda_device)
    image = ops.stitch(tiles_d, overlap)
    assert not image.is_contiguous() and ops.image_pitch(image) % 8 == 0
    want = o_st.stitch(tiles, overlap)
    np.testing.assert_array_equal(ops.to_host_dense(image, non_blocking=False).numpy(), want)
    np.testing.assert_array_equal(image.cpu().numpy(), want)
    if h <= 128:   # flat-field on the small cases (the oracle is slow at 2048^2 x 9)
        flat = 0.7 + 0.6 * rng.random((h, w))
        dark = 90.0 + 20 * rng.random((h, w))
        want_ff = o_st.stitch(o_ff.flatfield_correct(tiles, flat, dark), overlap)
        got_ff = ops.flatfield_stitch(tiles_d, flat, dark, overlap=overlap)
        np.testing.assert_array_equal(got_ff.cpu().numpy(), want_ff)
        image, want = got_ff, want_ff
    length, m = 40, 23
    x = rng.uniform(-5, wim + 5, (m, t))
    y = rng.uniform(-5, him + 5, (m, t))
    fg = rng.random((m, 1, length, length)) < 0.3
    bg = ~fg
    boxes = ops.bounding_boxes(dev(x, cuda_device), dev(y, cuda_device), length, wim, him)
    roi, stats = ops.roi_gather_stats(image, boxes, dev(fg.view(np.uint8), cuda_device), dev(bg.view(np.uint8), cuda_device), length)
    want_roi = o_rois.gather_rois(want, x, y, length)
    np.testing.assert_array_equal(roi.cpu().numpy(), want_roi)
    np.testing.assert_allclose(stats.cpu().numpy(), o_red.masked_stats(want_roi, np.repeat(fg, t, 1), np.repeat(bg, t, 1)),
                               rtol=1e-12, equal_nan=True)
    np.testing.assert_array_equal(ops.roi_gather(image, boxes, length).cpu().numpy(), want_roi)


def test_random_geometry_sweep(cuda_device):
    """Random tile grids, tile sizes and overlaps (every alignment class of the kept width, the
    clip and the image pitch): plain stitch for three dtypes and flat-field + stitch, all bit-exact
    against the oracle, dense and x-padded output images alike."""
    from magnify_b200 import ops

    rng = np.random.default_rng(2024)
    for trial in range(48):
        c, t, r, cc = (int(v) for v in rng.integers(1, 4, 4))
        h = int(rng.integers(9, 80))
        w = int(rng.choice([8, 16, 24, 40, 64, 72, 80])) if trial % 3 else int(rng.integers(9, 80))
        overlap = int(rng.integers(0, min(h, w) - 1))
        shape = (c, t, r, cc, h, w)
        dtype = [np.uint16, np.uint8, np.float32][trial % 3]
        tiles = (rng.random(shape) * 250).astype(dtype)
        want = o_st.stitch(tiles, overlap)
        got = ops.stitch(dev(tiles, cuda_device), overlap)
        np.testing.assert_array_equal(got.cpu().numpy(), want, err_msg=f"stitch {shape} ov {overlap} {dtype}")
        padded = ops.alloc_image(want.shape, got.dtype, cuda_device)
        ops.stitch(dev(tiles, cuda_device), overlap, out=padded)
        np.testing.assert_array_equal(ops.to_host_dense(padded, non_blocking=False).numpy(), want)
        if dtype == np.uint16:
            tiles16, flat, dark = _ff_case(rng, shape, per_channel=bool(trial % 2), scalar_dark=bool(trial % 4 == 0))
            want_ff = o_st.stitch(o_ff.flatfield_correct(tiles16, flat, dark), overlap)
            plan = ops.FlatFieldPlan(shape, flat, dark, device=cuda_device)
            out = ops.alloc_image(want_ff.shape, torch.uint16, cuda_device)
            ops.flatfield_stitch(dev(tiles16, cuda_device), overlap=overlap, plan=plan, out=out)
            np.testing.assert_array_equal(ops.to_host_dense(out, non_blocking=False).numpy(), want_ff,
                                          err_msg=f"flat-field {shape} ov {overlap}")


def test_random_gather_sweep(cuda_device):
    """Random window lengths (every parity / alignment class), image sizes (dense and x-padded),
    marker counts, mask timesteps and marker orders: crops bit-exact, masked sums exact, medians
    exact, for centres anywhere in and slightly beyond the image (boxes shift inwards, utils.py:66-80)."""
    from magnify_b200 import ops

    rng = np.random.default_rng(77)
    for trial in range(36):
        length = int(rng.integers(2, 110))
        c, t = int(rng.integers(1, 4)), int(rng.integers(1, 5))
        h, w = int(rng.integers(length, length + 200)), int(rng.integers(length, length + 260))
        m = int(rng.integers(1, 40))
        image = rng.integers(0, 65535, (c, t, h, w), dtype=np.uint16, endpoint=True)
        x = rng.uniform(-5, w + 5, (m, t))
        y = rng.uniform(-5, h + 5, (m, t))
        tm = int(rng.integers(1, t + 1))
        mask_t = np.sort(rng.integers(0, tm, t)).astype(np.int32)
        fg = rng.random((m, tm, length, length)) < rng.uniform(0, 1)
        bg = rng.random((m, tm, length, length)) < rng.uniform(0, 1)
        want_roi = o_rois.gather_rois(image, x, y, length)
        want = o_red.masked_stats(want_roi, fg[:, mask_t], bg[:, mask_t])
        img_d = ops.alloc_image(image.shape, torch.uint16, cuda_device) if trial % 2 else dev(image, cuda_device)
        if trial % 2:
            img_d.copy_(dev(image, cuda_device))
        boxes = ops.bounding_boxes(dev(x, cuda_device), dev(y, cuda_device), length, w, h)
        order = ops.spatial_order(boxes) if trial % 3 == 0 else None
        roi, stats = ops.roi_gather_stats(img_d, boxes, dev(fg.view(np.uint8), cuda_device), dev(bg.view(np.uint8), cuda_device),
                                          length, mask_t=dev(mask_t, cuda_device), order=order)
        msg = f"trial {trial}: L={length} image {(c, t, h, w)} m={m} tm={tm}"
        np.testing.assert_array_equal(roi.cpu().numpy(), want_roi, err_msg=msg)
        np.testing.assert_allclose(stats.cpu().numpy(), want, rtol=1e-12, equal_nan=True, err_msg=msg)
        np.testing.assert_array_equal(ops.roi_gather(img_d, boxes, length).cpu().numpy(), want_roi, err_msg=msg)
        med = ops.roi_median(roi, dev(fg.view(np.uint8), cuda_device), mask_t=dev(mask_t, cuda_device)).cpu().numpy()
        np.testing.assert_array_equal(med, o_red.masked_median(want_roi, fg[:, mask_t]), err_msg=msg)


def test_float32_roi_stats_and_float32_median(cuda_device):
    """The reductions on a float32 roi (the reference accepts float images): float64 sums in a
    fixed order (rtol 1e-12 against NumPy's float64 sums), exact medians (the two middle values
    of an even count averaged in float32, like np.nanmedian of the float32 roi), NaN pixels and
    empty masks handled like nanmean / nanmedian."""
    from magnify_b200 import ops

    rng = np.random.default_rng(31)
    for length in (5, 24, 72, 101):
        m, c, t = 7, 2, 3
        roi = (rng.standard_normal((m, c, t, length, length)) * 500 + 1000).astype(np.float32)
        roi[1, 0, 0, :2] = np.nan
        roi[2, 1, 1] = -3.5
        roi[3, 0, 2, 0, 0] = np.inf
        fg = rng.random((m, 2, length, length)) < 0.4
        bg = rng.random((m, 2, length, length)) < 0.6
        fg[4] = False
        mask_t = np.array([0, 1, 1], dtype=np.int32)
        stats = ops.roi_stats(dev(roi, cuda_device), dev(fg.view(np.uint8), cuda_device), dev(bg.view(np.uint8), cuda_device),
                              mask_t=dev(mask_t, cuda_device)).cpu().numpy()
        med = ops.roi_median(dev(roi, cuda_device), dev(fg.view(np.uint8), cuda_device), mask_t=dev(mask_t, cuda_device)).cpu().numpy()
        r64 = roi.astype(np.float64)
        for mi in range(m):
            for ci in range(c):
                for ti in range(t):
                    f, b = fg[mi, mask_t[ti]], bg[mi, mask_t[ti]]
                    px = r64[mi, ci, ti]
                    ok = ~np.isnan(px)
                    want = [float((f & ok).sum()), float((b & ok).sum()), px[f & ok].sum(), px[b & ok].sum()]
                    np.testing.assert_allclose(stats[mi, ci, ti, :4], want, rtol=1e-12)
                    with np.errstate(invalid="ignore", divide="ignore"):
                        means = [np.float64(want[2]) / want[0], np.float64(want[3]) / want[1]]
                    np.testing.assert_allclose(stats[mi, ci, ti, 4:6], means, rtol=1e-12, equal_nan=True)
                    vals = np.sort(roi[mi, ci, ti][f & ok])
                    if len(vals) == 0:
                        assert np.isnan(med[mi, ci, ti]) and np.isnan(stats[mi, ci, ti, 6])
                    else:
                        # `where` keeps the float32 roi float32: the two middle values are averaged
                        # in float32, as np.nanmedian does
                        lo, hi = vals[(len(vals) - 1) // 2], vals[len(vals) // 2]
                        want_med = np.float64(lo if len(vals) % 2 else (lo + hi) / np.float32(2))
                        assert want_med == np.float64(np.median(vals)), (length, mi, ci, ti)
                        assert med[mi, ci, ti] == want_med, (length, mi, ci, ti)
                        assert stats[mi, ci, ti, 6] == med[mi, ci, ti]


# ------------------------------------------------------- fused medians, hardened reductions
def _disc_masks(rng, m, tm, length, r_fg, r_in, r_out):
    yy, xx = np.mgrid[0:length, 0:length]
    fg = np.zeros((m, tm, length, length), dtype=bool)
    bg = np.zeros_like(fg)
    for i in range(m):
        for k in range(tm):
            cy, cx = rng.integers(length // 2 - 3, length // 2 + 4, 2)
            d2 = (yy - cy) ** 2 + (xx - cx) ** 2
            r = rng.integers(max(1, r_fg - 4), r_fg + 1)
            fg[i, k] = d2 <= r * r
            bg[i, k] = (d2 > r_in * r_in) & (d2 <= r_out * r_out)
    return fg, bg


@pytest.mark.parametrize("layout", ["cta", "warp"])
@pytest.mark.parametrize("length,r_fg,r_in,r_out", [(72, 15, 15, 30), (50, 10, 12, 24), (64, 14, 0, 26), (33, 6, 7, 15),
                                                      (100, 17, 20, 28)])
def test_gather_fused_medians(cuda_device, monkeypatch, layout, length, r_fg, r_in, r_out):
    """Masks small enough for the in-kernel value lists (chip discs / annuli, bead-sized masks):
    counts, sums, means and both medians come out of the gather itself, in both work layouts
    (one CTA per marker, one warp per marker) and with or without the crops; they equal the
    oracle's nanmean / nanmedian (identify.py:76-80, filter.py:21-22) exactly."""
    from magnify_b200 import ops

    monkeypatch.setenv("MGB_GATHER_LAYOUT", "1" if layout == "warp" else "0")
    rng = np.random.default_rng(length)
    c, t, h, w, m = 3, 4, 300, 512, 37
    image = np.clip(rng.normal(600, 40, (c, t, h, w)), 0, 65535).astype(np.uint16)
    image[0, 0, :40] = 65535                      # saturated band
    image[1] //= 64                               # few distinct values: many ties around the median
    x = rng.uniform(-5, w + 5, (m, t))
    y = rng.uniform(-5, h + 5, (m, t))
    mask_t = np.array([0, 1, 1, 0], dtype=np.int32)
    fg, bg = _disc_masks(rng, m, 2, length, r_fg, r_in, r_out)
    fg[3] = False                                 # empty masks -> NaN mean and median
    bg[4, 1] = False
    fg[5, 0] = False
    fg[5, 0, 10, 10] = True                       # single pixel
    fg[6, 0] = False
    fg[6, 0, 10, 10:12] = True                    # two pixels: mean of both
    want_roi = o_rois.gather_rois(image, x, y, length)
    want = o_red.masked_stats(want_roi, fg[:, mask_t], bg[:, mask_t])
    boxes = ops.bounding_boxes(dev(x, cuda_device), dev(y, cuda_device), length, w, h)
    fg_d, bg_d = dev(fg.view(np.uint8) * 255, cuda_device), dev(bg.view(np.uint8), cuda_device)   # 0/255 and 0/1 bytes
    counts = ops.mask_count_max(fg_d, bg_d)
    assert counts == (int(fg.sum((-1, -2)).max()), int(bg.sum((-1, -2)).max()))
    for want_roi_flag in (True, False):
        roi, stats = ops.roi_gather_stats(dev(image, cuda_device), boxes, fg_d, bg_d, length,
                                          mask_t=dev(mask_t, cuda_device), want_roi=want_roi_flag, mask_counts=counts)
        if want_roi_flag:
            np.testing.assert_array_equal(roi.cpu().numpy(), want_roi)
        got = stats.cpu().numpy()
        np.testing.assert_array_equal(got[..., :4], want[..., :4])
        np.testing.assert_allclose(got[..., 4:6], want[..., 4:6], rtol=1e-12, equal_nan=True)
        np.testing.assert_array_equal(got[..., 6:], want[..., 6:])
    _, no_med = ops.roi_gather_stats(dev(image, cuda_device), boxes, fg_d, bg_d, length, mask_t=dev(mask_t, cuda_device),
                                     medians=False, mask_counts=counts)
    no_med = no_med.cpu().numpy()
    np.testing.assert_array_equal(no_med[..., :6], got[..., :6])
    assert np.isnan(no_med[..., 6:]).all()


_SPLIT_TAILS = [(9, None, False)] + [(k, w, True) for k in (1, 9, "third", "last") for w in (6, 12)]


@pytest.mark.parametrize("tail", _SPLIT_TAILS, ids=[f"k{k}-w{w or 'auto'}-{'perm' if o else 'id'}" for k, w, o in _SPLIT_TAILS])
@pytest.mark.parametrize("c,t", [(3, 10), (4, 33)])
def test_gather_split_last_wave(cuda_device, monkeypatch, c, t, tail):
    """A few more markers than a multiple of the resident CTAs: the markers of the last, nearly
    empty wave are shared by several CTAs each (roi_lists.cu).  Same crops and summaries as the
    oracle and as the unsplit launch, with few windows per marker (two 6-warp CTAs per SM) and
    with many (one 12-warp CTA).  tail = (k, warps, order): M = 2 x SMs + k markers for k = 1, 9,
    SMs / 3 ("third") and SMs - 1 ("last"), at 6 or 12 warps per CTA, with the markers in a random
    processing order (the split deals marker slots, which `order` then maps to markers)."""
    from magnify_b200 import ops

    sms = torch.cuda.get_device_properties(cuda_device).multi_processor_count
    k, warps, shuffle = tail
    k = {"third": sms // 3, "last": sms - 1}.get(k, k)
    m, length, h, w = 2 * sms + k, 33, 200, 320
    rng = np.random.default_rng(c * 100 + t)
    image = np.clip(rng.normal(700, 60, (c, t, h, w)), 0, 65535).astype(np.uint16)
    x = rng.uniform(0, w, (m, t))
    y = rng.uniform(0, h, (m, t))
    fg, bg = _disc_masks(rng, m, 1, length, 6, 7, 15)
    want_roi = o_rois.gather_rois(image, x, y, length)
    want = o_red.masked_stats(want_roi, np.repeat(fg, t, 1), np.repeat(bg, t, 1))
    boxes = ops.bounding_boxes(dev(x, cuda_device), dev(y, cuda_device), length, w, h)
    fg_d, bg_d = dev(fg.view(np.uint8), cuda_device), dev(bg.view(np.uint8), cuda_device)
    counts = ops.mask_count_max(fg_d, bg_d)
    order = dev(rng.permutation(m).astype(np.int32), cuda_device) if shuffle else None
    monkeypatch.setenv("MGB_GATHER_LAYOUT", "0")
    if warps:
        monkeypatch.setenv("MGB_GATHER_WARPS", str(warps))
    else:
        monkeypatch.delenv("MGB_GATHER_WARPS", raising=False)
    results = []
    for split in ("1", "0"):
        monkeypatch.setenv("MGB_GATHER_SPLIT", split)
        roi, stats = ops.roi_gather_stats(dev(image, cuda_device), boxes, fg_d, bg_d, length, mask_counts=counts,
                                          order=order)
        assert ops.last_gather_fused is True
        np.testing.assert_array_equal(roi.cpu().numpy(), want_roi)
        got = stats.cpu().numpy()
        np.testing.assert_array_equal(got[..., :4], want[..., :4])
        np.testing.assert_allclose(got[..., 4:6], want[..., 4:6], rtol=1e-12, equal_nan=True)
        np.testing.assert_array_equal(got[..., 6:], want[..., 6:])
        results.append(got)
    np.testing.assert_array_equal(results[0], results[1])


@pytest.mark.parametrize("length", [256, 300, 1024])
def test_saturated_sums_do_not_wrap(cuda_device, gather_path, length):
    """A 65535-valued image under full masks: the per-ROI sums (L^2 * 65535, above 2^32 from
    L = 257) must be exact in every gather kernel, also with 255-valued mask bytes."""
    from magnify_b200 import ops

    c, t, h, w, m = 1, 2, length + 8, length + 16, 3
    image = torch.full((c, t, h, w), 65535, dtype=torch.uint16, device=cuda_device)
    x = torch.tensor([[length / 2, length / 2 + 3.0]] * m, dtype=torch.float64, device=cuda_device)
    y = torch.tensor([[length / 2 + 1.0, length / 2]] * m, dtype=torch.float64, device=cuda_device)
    boxes = ops.bounding_boxes(x, y, length, w, h)
    fg = torch.full((m, 1, length, length), 255, dtype=torch.uint8, device=cuda_device)
    bg = torch.ones((m, 1, length, length), dtype=torch.uint8, device=cuda_device)
    bg[1, 0, ::2] = 0
    roi, stats = ops.roi_gather_stats(image, boxes, fg, bg, length)
    assert bool((roi == 65535).all())
    s = stats.cpu().numpy()
    n_bg = bg.sum((-1, -2, -3)).cpu().numpy().astype(np.float64)
    np.testing.assert_array_equal(s[..., 0], float(length * length))
    np.testing.assert_array_equal(s[..., 2], float(length * length) * 65535.0)
    np.testing.assert_array_equal(s[..., 1], np.broadcast_to(n_bg[:, None, None], s[..., 1].shape))
    np.testing.assert_array_equal(s[..., 3], np.broadcast_to(n_bg[:, None, None] * 65535.0, s[..., 3].shape))
    np.testing.assert_array_equal(s[..., 4:], 65535.0)
    stats2 = ops.roi_stats(roi, fg, bg).cpu().numpy()
    np.testing.assert_array_equal(stats2, s)


@pytest.mark.parametrize("length", [161, 200, 333])
def test_median_large_roi(cuda_device, length):
    """roi_length above 160 (max_bead_diameter > 80 gives L = 2 d; chamber_diameter > 133 gives
    L = 1.2 d): the median re-reads the window per bisection step instead of refusing."""
    from magnify_b200 import ops

    rng = np.random.default_rng(length)
    m, c, t = 3, 2, 2
    roi = rng.integers(0, 65535, (m, c, t, length, length), dtype=np.uint16, endpoint=True)
    roi[1] //= 4096
    mask = rng.random((m, t, length, length)) < 0.5
    mask[2, 1] = False
    got = ops.roi_median(dev(roi, cuda_device), dev(mask.view(np.uint8), cuda_device)).cpu().numpy()
    np.testing.assert_array_equal(got, o_red.masked_median(roi, mask))
    f32 = (rng.standard_normal((m, c, t, length, length)) * 100).astype(np.float32)
    got = ops.roi_median(dev(f32, cuda_device), dev(mask.view(np.uint8), cuda_device)).cpu().numpy()
    np.testing.assert_array_equal(got, o_red.masked_median(f32, mask))


def test_identity_flatfield_on_float_tiles_still_clips(cuda_device):
    """flat = 1, dark = 0 is only the identity for unsigned integers: the reference still runs
    clip(min=0) and (x * M) / M on float tiles (preprocess.py:83-87), which zeroes negative pixels."""
    from magnify_b200 import ops

    rng = np.random.default_rng(5)
    for dtype in (np.float32, np.float64):
        tiles = (rng.standard_normal((2, 1, 2, 2, 24, 32)) * 100).astype(dtype)
        want_tiles = o_ff.flatfield_correct(tiles, 1.0, 0.0)
        assert (want_tiles >= 0).all() and (tiles < 0).any()
        got = ops.flatfield_correct(dev(tiles, cuda_device), 1.0, 0.0).cpu().numpy()
        np.testing.assert_array_equal(got, want_tiles)
        got = ops.flatfield_stitch(dev(tiles, cuda_device), 1.0, 0.0, overlap=4).cpu().numpy()
        np.testing.assert_array_equal(got, o_st.stitch(want_tiles, 4))
    u16 = rng.integers(0, 65535, (1, 1, 2, 2, 16, 16), dtype=np.uint16, endpoint=True)
    np.testing.assert_array_equal(ops.flatfield_correct(dev(u16, cuda_device), 1.0, 0.0).cpu().numpy(), u16)
