"""The reference-facing components (magnify_b200.components) on the Assay stand-in: same
arguments, exceptions and dataset schema as the reference's Stitcher / flatfield_correct /
BeadFinder / ButtonFinder, pixel values against the oracle and the golden fixtures."""
import numpy as np
import pytest
import torch

from oracle import flatfield as o_ff
from oracle import reduce as o_red
from oracle import stitch as o_st

pytestmark = pytest.mark.gpu

TILE_DIMS = ("channel", "time", "tile_row", "tile_col", "tile_y", "tile_x")


def tile_assay(tile_data):
    from magnify_b200.dataset import Assay

    return Assay({"tile": (TILE_DIMS, tile_data)})


# ---- port of the reference's tests/test_stitch.py against the component ----------------------
def test_stitcher_basic(cuda_device):  # tests/test_stitch.py:9-26
    from magnify_b200.components import Stitcher

    tile_data = np.random.rand(1, 1, 2, 3, 40, 40)
    result = Stitcher(overlap=5)(tile_assay(tile_data))
    assert "image" in result.data_vars
    assert result.sizes["im_y"] == 2 * (40 - 5)
    assert result.sizes["im_x"] == 3 * (40 - 5)
    np.testing.assert_array_equal(result.image[0, 0, 35:70, 35:70], tile_data[0, 0, 1, 1, 2:37, 2:37])


def test_stitcher_single_tile_and_zero_overlap(cuda_device):  # :28-45, :78-96
    from magnify_b200.components import Stitcher

    tile_data = np.random.rand(1, 1, 1, 1, 30, 30)
    result = Stitcher(overlap=5)(tile_assay(tile_data))
    assert result.sizes["im_y"] == 25 and result.sizes["im_x"] == 25
    np.testing.assert_array_equal(result.image[0, 0], tile_data[0, 0, 0, 0, 2:27, 2:27])
    tile_data = np.random.rand(1, 1, 1, 2, 20, 20)
    result = Stitcher(overlap=0)(tile_assay(tile_data))
    assert result.sizes["im_y"] == 20 and result.sizes["im_x"] == 40
    np.testing.assert_array_equal(result.image[0, 0, :, :20], tile_data[0, 0, 0, 0])
    np.testing.assert_array_equal(result.image[0, 0, :, 20:], tile_data[0, 0, 0, 1])


def test_stitcher_preserves_channels_and_time(cuda_device):  # :47-76
    from magnify_b200.components import Stitcher

    result = Stitcher(overlap=8)(tile_assay(np.random.rand(2, 3, 2, 2, 25, 25)))
    assert result.image.dims == ("channel", "time", "im_y", "im_x")
    assert result.sizes["channel"] == 2 and result.sizes["time"] == 3


def test_stitcher_errors(cuda_device):  # :98-125
    from magnify_b200.components import Stitcher
    from magnify_b200.dataset import Assay

    with pytest.raises(ValueError):
        Stitcher(overlap=-5)
    with pytest.raises(AttributeError):
        Stitcher(overlap=10)(Assay({"other_data": (("x",), np.array([1, 2, 3]))}))
    with pytest.raises(ValueError):
        Stitcher(overlap=100)(tile_assay(np.random.rand(1, 1, 2, 2, 50, 50)))


# ---- flat-field ------------------------------------------------------------------------------
def test_flatfield_components(cuda_device):
    from magnify_b200.components import FlatfieldStitcher, Stitcher, flatfield_correct

    rng = np.random.default_rng(0)
    tiles = np.clip(rng.normal(2000, 800, (2, 2, 2, 2, 64, 64)), 0, 65535).astype(np.uint16)
    flat = 0.7 + 0.6 * rng.random((64, 64))
    dark = 90.0 + 10 * rng.random((64, 64))
    want_tiles = o_ff.flatfield_correct(tiles, flat, dark)
    xp = flatfield_correct(tile_assay(tiles.copy()), flatfield=flat, darkfield=dark)
    np.testing.assert_array_equal(xp.tile.values, want_tiles)
    xp = Stitcher(overlap=6)(xp)
    np.testing.assert_array_equal(xp.image.values, o_st.stitch(want_tiles, 6))
    fused = FlatfieldStitcher(flat, dark, overlap=6)(tile_assay(tiles.copy()))
    np.testing.assert_array_equal(fused.image.values, o_st.stitch(want_tiles, 6))
    # defaults are the identity (registry.py:278-279)
    xp = flatfield_correct(tile_assay(tiles.copy()))
    np.testing.assert_array_equal(xp.tile.values, tiles)


# ---- find_beads / find_buttons ---------------------------------------------------------------
def test_bead_finder_schema_and_values(cuda_device, golden, make_pattern_image):
    from magnify_b200.components import BeadFinder, quantify
    from magnify_b200.dataset import Assay

    g = golden("beads")
    c, t, h, w = (int(v) for v in g["image_shape"])
    image = make_pattern_image(c, t, h, w, salt=int(g["image_salt"]))
    assay = Assay({"image": (("channel", "time", "im_y", "im_x"), image)},
                  coords={"channel": (("channel",), np.array(["a", "b"]))})
    finder = BeadFinder(min_bead_diameter=2, max_bead_diameter=50, roi_length=int(g["roi_length"]), centers=g["beads"])
    out = finder(assay)
    assert out.roi.dims == ("mark", "channel", "time", "roi_y", "roi_x")          # find.py:533
    assert out.fg.dims == ("mark", "time", "roi_y", "roi_x") and out.fg.dtype == bool
    assert out.x.dims == ("mark", "time") and out.valid.dtype == bool
    np.testing.assert_array_equal(out.roi.values, g["roi"])
    np.testing.assert_array_equal(out.fg.values, np.repeat(g["fg"][:, None], t, 1))
    np.testing.assert_array_equal(out.bg.values, np.repeat(g["bg"][:, None], t, 1))
    np.testing.assert_array_equal(out.x.values[:, 0], g["beads"][:, 1])
    np.testing.assert_array_equal(out.y.values[:, 0], g["beads"][:, 0])
    assert out.valid.values.all()
    q = quantify(out)
    fgt, bgt = np.repeat(g["fg"][:, None], t, 1), np.repeat(g["bg"][:, None], t, 1)
    want = o_red.masked_stats(g["roi"], fgt, bgt)
    np.testing.assert_allclose(q.fg_mean.values, want[..., 4], rtol=1e-12, equal_nan=True)
    np.testing.assert_allclose(q.bg_mean.values, want[..., 5], rtol=1e-12, equal_nan=True)
    np.testing.assert_array_equal(q.bg_median.values, o_red.masked_median(g["roi"], bgt))
    # identify.py:76-80: mean(fg) - median(bg)
    intensity = q.fg_mean.values - q.bg_median.values
    assert intensity.shape == (len(g["beads"]), c, t)
    with pytest.raises(ValueError):
        BeadFinder(min_bead_diameter=30, max_bead_diameter=10)                     # find.py:458-459


def test_bead_finder_no_beads(cuda_device):  # find.py:557-558, tests/test_beads.py:219-232
    from magnify_b200.components import BeadFinder
    from magnify_b200.dataset import Assay

    assay = Assay({"image": (("channel", "time", "im_y", "im_x"), np.zeros((1, 1, 128, 128), np.uint16))})
    out = BeadFinder(16, 24, centers=np.empty((0, 3)))(assay)
    assert out.sizes["mark"] == 0 and out.roi.shape == (0, 1, 1, 48, 48)


def test_button_finder_schema_and_values(cuda_device, golden, make_pattern_image):
    from magnify_b200.components import ButtonFinder
    from magnify_b200.dataset import Assay

    g = golden("chip")
    c, t, h, w = (int(v) for v in g["image_shape"])
    image = make_pattern_image(c, t, h, w, salt=int(g["image_salt"]))
    rows, cols = g["x"].shape
    assay = Assay({"image": (("channel", "time", "im_y", "im_x"), image)},
                  coords={"tag": (("mark_row", "mark_col"), np.full((rows, cols), "default")),
                          "valid": (("mark_row", "mark_col", "time"), np.ones((rows, cols, t), bool))})

    def centers(assay, ts):   # pinned outcome of the CPU centre search + refinement at timestep ts
        assert ts == 0
        return g["x"], g["y"], g["fg_radius"]

    finder = ButtonFinder(row_dist=100, col_dist=150, min_button_diameter=16, max_button_diameter=30,
                          chamber_diameter=60, search_timestep=0, centers=centers)
    assert finder.roi_length == 72 and finder.chamber_radius == 30 and finder.max_button_radius == 15
    out = finder(assay)
    np.testing.assert_array_equal(out.roi.values, g["roi"])
    np.testing.assert_array_equal(out.fg.values, g["fg"])
    np.testing.assert_array_equal(out.bg.values, g["bg"])
    # copy-forward: identical x, y on non-searched timesteps (tests/test_chip.py:449-456)
    for ti in range(1, t):
        np.testing.assert_array_equal(out.x.values[:, ti], out.x.values[:, 0])
        np.testing.assert_array_equal(out.y.values[:, ti], out.y.values[:, 0])
    assert out.tag.dims == ("mark",) and out.valid.dims == ("mark", "time")
    with pytest.raises(ValueError):
        ButtonFinder(100, 100, 30, 10, 60)                                          # find.py:34-35


def test_button_finder_multi_search_matches_reference_call(cuda_device, golden, make_pattern_image):
    """tests/golden/chip_multi.npz is the output of the reference's own ButtonFinder.__call__ with
    search_timestep=[1, 3] (executed in place, centre search pinned): the component must give the
    same roi / fg / bg / x / y, including the copy-forward of find.py:143-181."""
    from magnify_b200.components import ButtonFinder
    from magnify_b200.dataset import Assay

    g = golden("chip_multi")
    c, t, h, w = (int(v) for v in g["image_shape"])
    image = make_pattern_image(c, t, h, w, salt=int(g["image_salt"]))
    rows, cols = g["coarse_x"].shape
    search = [int(v) for v in g["search_timesteps"]]
    refine = g["refine"].reshape(len(search), rows, cols, 3)
    radius = np.where(refine[..., 2] >= 0, refine[..., 2], int(g["max_button_radius"]))
    assay = Assay({"image": (("channel", "time", "im_y", "im_x"), image)},
                  coords={"tag": (("mark_row", "mark_col"), np.full((rows, cols), "default")),
                          "valid": (("mark_row", "mark_col", "time"), np.ones((rows, cols, t), bool))})

    def centers(assay, ts):
        k = search.index(ts)
        return g["x"][:, ts].reshape(rows, cols), g["y"][:, ts].reshape(rows, cols), radius[k]

    finder = ButtonFinder(row_dist=100, col_dist=150, min_button_diameter=8, max_button_diameter=18,
                          chamber_diameter=34, roi_length=int(g["roi_length"]), search_timestep=search, centers=centers)
    out = finder(assay)
    np.testing.assert_array_equal(out.roi.values, g["roi"])
    np.testing.assert_array_equal(out.fg.values, g["fg"])
    np.testing.assert_array_equal(out.bg.values, g["bg"])
    np.testing.assert_array_equal(out.x.values, g["x"])
    np.testing.assert_array_equal(out.y.values, g["y"])


def test_finders_with_pinned_centres_never_synchronise(cuda_device):
    """ButtonFinder and BeadFinder with pinned centres on the stitched image in HBM only queue
    work: no synchronising copy or read-back, so an assay's finder never waits behind its image
    download and the next assay's upload can be queued at once."""
    from magnify_b200.components import BeadFinder, ButtonFinder, Stitcher
    from magnify_b200.dataset import Assay
    from oracle import rois as o_rois
    from test_gpu_end_to_end import split_into_tiles
    from test_gpu_finders import draw_chip

    rows, cols, t, overlap = 3, 4, 3, 8
    chip = draw_chip((rows, cols), 20, row_dist=100, col_dist=100) + 50                     # (400, 500)
    tiles = np.stack([split_into_tiles(chip + 3 * k, 2, 2, overlap) for k in range(t)])[None]
    xp = Stitcher(overlap, device=cuda_device)(Assay({"tile": (TILE_DIMS, tiles)},
                                                     coords={"tag": (("mark_row", "mark_col"), np.full((rows, cols), "a"))}))
    image = xp["image"].data
    yy, xx = np.mgrid[1:rows + 1, 1:cols + 1] * 100.0

    def centers(assay, ts):
        return xx + ts, yy - ts, np.full((rows, cols), 10)

    beads = np.array([[100.0, 100.0, 10.0], [200.0, 300.0, 10.0], [310.0, 420.0, 9.0]])
    bead_assay = Assay({"image": (("channel", "time", "im_y", "im_x"), image)})
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        chips = ButtonFinder(100, 100, 16, 32, 60, search_timestep=[0, 2], centers=centers, device=cuda_device)(xp)
        found = BeadFinder(16, 24, centers=beads, device=cuda_device)(bead_assay)
    finally:
        torch.cuda.set_sync_debug_mode("default")
    host = image.numpy()
    x, y = chips.x.values, chips.y.values
    assert (x[:, 1] == x[:, 0]).all() and (x[:, 2] == x[:, 0] + 2).all()                  # copied forward from t = 0
    np.testing.assert_array_equal(chips.roi.values, o_rois.gather_rois(host, x, y, 72))
    np.testing.assert_array_equal(found.roi.values, o_rois.gather_rois(host, found.x.values, found.y.values, 48))


def test_filter_expression_and_mrbles_intensities(cuda_device):
    """SURVEY.md section 8f row N3: the consumers of the summaries (filter.py:11-37,
    identify.py:76-80) on GPU medians / means, against the NumPy restatement."""
    from magnify_b200.components import filter_expression, mrbles_intensities
    from magnify_b200.dataset import Assay

    rng = np.random.default_rng(17)
    m, c, t, length = 40, 3, 2, 24
    roi = rng.integers(380, 420, (m, c, t, length, length)).astype(np.uint16)
    yy, xx = np.mgrid[0:length, 0:length]
    fg0 = (yy - 12) ** 2 + (xx - 12) ** 2 <= 25
    fg = np.broadcast_to(fg0, (m, t, length, length)).copy()
    bg = ~np.broadcast_to((yy - 12) ** 2 + (xx - 12) ** 2 <= 64, (m, t, length, length))
    roi[: m // 2, 1][:, :, fg0] += 300            # half of the markers are expressed in channel 1
    valid = np.ones((m, t), bool)
    valid[3] = False
    assay = Assay({"roi": (("mark", "channel", "time", "roi_y", "roi_x"), roi)},
                  coords={"fg": (("mark", "time", "roi_y", "roi_x"), fg), "bg": (("mark", "time", "roi_y", "roi_x"), bg),
                          "valid": (("mark", "time"), valid), "channel": (("channel",), np.array(["a", "b", "c"]))})
    out = filter_expression(assay, search_channel="b")
    want = o_red.filter_expression_valid(roi, fg, bg, valid, channels=[1])
    np.testing.assert_array_equal(out.valid.values, want)
    assert want[: m // 2].sum() >= (m // 2 - 1) * t and not want[m // 2 :].any()
    out2 = filter_expression(assay, min_contrast=1000)
    np.testing.assert_array_equal(out2.valid.values, o_red.filter_expression_valid(roi, fg, bg, valid, [0, 1, 2], 1000))
    inten = mrbles_intensities(assay, channels=["a", "b"])
    np.testing.assert_allclose(inten, o_red.mrbles_intensities(roi[:, :2], fg, bg), rtol=1e-12)


def test_filter_expression_golden_from_reference_source(cuda_device, golden):
    """GPU medians + the reference's threshold logic against tests/golden/filter.npz (outputs of the
    reference's own filter_expression source, filter.py:11-37, executed in place)."""
    from magnify_b200.components import filter_expression
    from magnify_b200.dataset import Assay

    g = golden("filter")
    names = [str(v) for v in g["channels"]]
    k = 0
    while f"case{k}__valid" in g:
        search = [str(v) for v in g[f"case{k}__search"]] or None
        mc = int(g[f"case{k}__min_contrast"])
        assay = Assay({"roi": (("mark", "channel", "time", "roi_y", "roi_x"), g["roi"])},
                      coords={"channel": (("channel",), np.array(names)),
                              "fg": (("mark", "time", "roi_y", "roi_x"), g["fg"]),
                              "bg": (("mark", "time", "roi_y", "roi_x"), g["bg"]),
                              "valid": (("mark", "time"), g["valid"])})
        out = filter_expression(assay, search_channel=search, min_contrast=None if mc < 0 else mc)
        np.testing.assert_array_equal(out.valid.values, g[f"case{k}__valid"], err_msg=f"case {k}")
        k += 1
    assert k == 6


def test_mrbles_intensities_golden_from_reference_expression(cuda_device, golden):
    """identify.py:76-80 run in place -> tests/golden/filter.npz; GPU mean/median must reproduce the
    float64 result to 1e-12 and the float32-promoted one to 1e-5 of the mean (north_star)."""
    from magnify_b200.components import mrbles_intensities
    from magnify_b200.dataset import Assay

    g = golden("filter")
    assay = Assay({"roi": (("mark", "channel", "time", "roi_y", "roi_x"), g["roi"])},
                  coords={"channel": (("channel",), np.array([str(v) for v in g["channels"]])),
                          "fg": (("mark", "time", "roi_y", "roi_x"), g["fg"]),
                          "bg": (("mark", "time", "roi_y", "roi_x"), g["bg"])})
    got = mrbles_intensities(assay, channels=[str(v) for v in g["intensity_channels"]])
    np.testing.assert_allclose(got, g["intensities_f64"], rtol=1e-12, atol=1e-10)
    np.testing.assert_allclose(got, g["intensities_f32"], rtol=0, atol=1e-5 * 500.0)
    assert np.isnan(got[7]).all()


def test_filter_leaky_golden_from_reference_source(cuda_device, golden):
    """GPU medians + the reference's neighbour logic against the outputs of the reference's own
    filter_leaky_buttons (filter.py:65-94) executed in place (tests/golden/filter.npz)."""
    from magnify_b200.components import filter_leaky
    from magnify_b200.dataset import Assay

    g = golden("filter")
    names = [str(v) for v in g["channels"]]
    for k in range(3):
        search = [str(v) for v in g[f"leaky{k}__search"]] or None
        assay = Assay({"roi": (("mark", "channel", "time", "roi_y", "roi_x"), g["roi"])},
                      coords={"channel": (("channel",), np.array(names)),
                              "fg": (("mark", "time", "roi_y", "roi_x"), g["fg"]),
                              "bg": (("mark", "time", "roi_y", "roi_x"), g["bg"]),
                              "tag": (("mark",), g["tag"]), "mark_row": (("mark",), g["mark_row"]),
                              "valid": (("mark", "time"), g["valid"])})
        out = filter_leaky(assay, search_channel=search)
        np.testing.assert_array_equal(out.valid.values, g[f"leaky{k}__valid"], err_msg=f"case {k}")


def test_mask_perimeters_match_opencv(cuda_device):
    """ops.mask_perimeters == sum of cv.arcLength over cv.findContours(RETR_EXTERNAL,
    CHAIN_APPROX_SIMPLE) (filter.py:54-55) on noise, rings with islands, discs and blobs."""
    cv2 = pytest.importorskip("cv2")
    from magnify_b200 import ops

    rng = np.random.default_rng(0)
    for length in (1, 2, 3, 7, 24, 48, 72, 100, 160, 161, 200, 333):    # above 160: int32 labels in a global workspace
        masks = []
        yy, xx = np.mgrid[0:length, 0:length]
        for trial in range(24 if length <= 160 else 8):
            kind = trial % 4
            if kind == 0:
                m = rng.random((length, length)) < rng.uniform(0.1, 0.9)
            elif kind == 1:
                d2 = (yy - length / 2) ** 2 + (xx - length / 2) ** 2
                m = (d2 <= (length / 3) ** 2) & ~(d2 <= (length / 6) ** 2) | (d2 <= (length / 12) ** 2)
            elif kind == 2:
                m = (yy - rng.uniform(0, length)) ** 2 + (xx - rng.uniform(0, length)) ** 2 <= rng.uniform(1, length / 2 + 1) ** 2
            else:
                m = cv2.GaussianBlur(rng.random((length, length)).astype(np.float32), (5, 5), 0) > 0.5
            masks.append(m)
        masks = np.stack(masks)
        masks[-1] = False
        got = ops.mask_perimeters(torch.from_numpy(masks).to(cuda_device)).cpu().numpy()
        want = []
        for m in masks:
            contours, _ = cv2.findContours(m.astype(np.uint8) * 255, cv2.RETR_EXTERNAL, cv2.CHAIN_APPROX_SIMPLE)
            want.append(sum(cv2.arcLength(c, True) for c in contours))
        np.testing.assert_allclose(got, want, rtol=1e-6, atol=0)
        assert got[-1] == 0


def test_filter_nonround_golden_from_reference_source(cuda_device, golden):
    from magnify_b200.components import filter_nonround
    from magnify_b200.dataset import Assay

    g = golden("nonround")
    for k in range(3):
        assay = Assay(coords={"fg": (("mark", "time", "roi_y", "roi_x"), g["fg"]), "valid": (("mark", "time"), g["valid"])})
        out = filter_nonround(assay, min_roundness=float(g[f"case{k}__min_roundness"]))
        np.testing.assert_array_equal(out.valid.values, g[f"case{k}__valid"], err_msg=f"case {k}")


def test_quantify_and_filters_accept_float_roi(cuda_device):
    """quantify / filter_expression on a float32 roi equal the uint16 run on the same values."""
    from magnify_b200.components import filter_expression, quantify
    from magnify_b200.dataset import Assay

    rng = np.random.default_rng(3)
    m, c, t, length = 20, 2, 2, 24
    roi = rng.integers(380, 420, (m, c, t, length, length)).astype(np.uint16)
    yy, xx = np.mgrid[0:length, 0:length]
    fg0 = (yy - 12) ** 2 + (xx - 12) ** 2 <= 25
    roi[::2][..., fg0] += 300
    fg = np.broadcast_to(fg0, (m, t, length, length)).copy()
    bg = np.broadcast_to((yy - 12) ** 2 + (xx - 12) ** 2 > 64, (m, t, length, length)).copy()

    def assay(values):
        return Assay({"roi": (("mark", "channel", "time", "roi_y", "roi_x"), values)},
                     coords={"channel": (("channel",), np.array(["a", "b"])), "fg": (("mark", "time", "roi_y", "roi_x"), fg),
                             "bg": (("mark", "time", "roi_y", "roi_x"), bg), "valid": (("mark", "time"), np.ones((m, t), bool))})

    a16, a32 = quantify(assay(roi)), quantify(assay(roi.astype(np.float32)))
    for name in ("fg_sum", "bg_sum", "fg_mean", "bg_mean", "fg_median", "bg_median", "fg_count"):
        np.testing.assert_array_equal(a16[name].values, a32[name].values, err_msg=name)
    v16 = filter_expression(assay(roi)).valid.values
    v32 = filter_expression(assay(roi.astype(np.float32))).valid.values
    np.testing.assert_array_equal(v16, v32)
    assert v16[::2].all() and v16[1::2].sum() < v16[::2].sum()     # the bright half is expressed
