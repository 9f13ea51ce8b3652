"""Oracle restatements of stitch / flat-field / ROI paths: the reference's own golden
assertions (tests/test_stitch.py) and the golden fixtures replayed from the real utils.py."""
import numpy as np
import pytest

from oracle import flatfield as ff
from oracle import reduce as red
from oracle import rois
from oracle import stitch as st


# ---- port of the reference's tests/test_stitch.py (array level) -------------------------------
def test_stitcher_basic():  # tests/test_stitch.py:9-26
    tile_data = np.random.rand(1, 1, 2, 3, 40, 40)
    image = st.stitch(tile_data, 5)
    assert image.shape[-2] == 2 * (40 - 5) and image.shape[-1] == 3 * (40 - 5)
    np.testing.assert_array_equal(image[0, 0, 35:70, 35:70], tile_data[0, 0, 1, 1, 2:37, 2:37])


def test_stitcher_single_tile():  # :28-45
    tile_data = np.random.rand(1, 1, 1, 1, 30, 30)
    image = st.stitch(tile_data, 5)
    assert image.shape[-2:] == (25, 25)
    np.testing.assert_array_equal(image[0, 0], tile_data[0, 0, 0, 0, 2:27, 2:27])


def test_stitcher_preserves_channels_and_time():  # :47-76
    image = st.stitch(np.random.rand(2, 3, 2, 2, 25, 25), 8)
    assert image.shape[:2] == (2, 3)


def test_stitcher_zero_overlap():  # :78-96
    tile_data = np.random.rand(1, 1, 1, 2, 20, 20)
    image = st.stitch(tile_data, 0)
    assert image.shape[-2:] == (20, 40)
    np.testing.assert_array_equal(image[0, 0, :, :20], tile_data[0, 0, 0, 0])
    np.testing.assert_array_equal(image[0, 0, :, 20:], tile_data[0, 0, 0, 1])


def test_stitcher_errors():  # :98-100, :112-125
    with pytest.raises(ValueError):
        st.check_overlap(-5)
    with pytest.raises(ValueError):
        st.stitch(np.random.rand(1, 1, 2, 2, 50, 50), 100)


STITCH_CASES = ("odd", "even", "zero", "single", "max")


def test_stitch_golden_from_reference_source(golden):
    """tests/golden/stitch.npz = outputs of the reference's own Stitcher source (stitch.py:12-46)."""
    g = golden("stitch")
    for name in STITCH_CASES:
        got = st.stitch(g[name + "__tiles"], int(g[name + "__overlap"]))
        assert got.dtype == g[name + "__image"].dtype
        np.testing.assert_array_equal(got, g[name + "__image"], err_msg=name)


STITCH_OVERLAPS = (0, 1, 4, 7, 13)


def stitch_tiles():
    return np.random.default_rng(3).integers(0, 65535, (2, 2, 3, 2, 14, 18), dtype=np.uint16, endpoint=True)


def flatfield_case():
    rng = np.random.default_rng(7)
    tiles = rng.integers(0, 65535, (2, 1, 2, 2, 16, 16), dtype=np.uint16, endpoint=True)
    flat = 0.6 + 0.8 * rng.random((16, 16))
    dark = 80 + 40 * rng.random((16, 16))
    return tiles, flat, dark


def record():
    """This package's side of the stitch and flat-field comparisons with the reference in this
    module (written to tests/golden/reference_record.npz by tests/golden/make_reference_record.py)."""
    tiles = stitch_tiles()
    out = {f"stitch_{ov}": st.stitch(tiles, ov) for ov in STITCH_OVERLAPS}
    out["flatfield"] = ff.flatfield_correct(*flatfield_case())
    return out


def test_stitch_against_reference_source_when_present(golden):
    """What the reference's Stitcher returned (tests/golden/reference_record.npz), and the
    reference itself when it is present."""
    from oracle._refload import reference_stitch

    rec, tiles = golden("reference_record"), stitch_tiles()
    for ov in STITCH_OVERLAPS:
        want = rec[f"stitch_{ov}"]
        np.testing.assert_array_equal(st.stitch(tiles, ov), want)
        ref = reference_stitch(tiles, ov)
        if ref is not None:
            np.testing.assert_array_equal(ref, want)


# ---- flat-field ------------------------------------------------------------------------------
def test_flatfield_defaults_are_identity():
    rng = np.random.default_rng(0)
    tiles = rng.integers(0, 65535, (2, 2, 1, 2, 16, 16), dtype=np.uint16, endpoint=True)
    np.testing.assert_array_equal(ff.flatfield_correct(tiles), tiles)


def test_flatfield_formula_and_chunked_maxima():
    rng = np.random.default_rng(1)
    tiles = rng.integers(0, 5000, (2, 2, 2, 2, 12, 16), dtype=np.uint16)
    flat = 0.7 + 0.6 * rng.random((12, 16))
    dark = 90 + 20 * rng.random((12, 16))
    out = ff.flatfield_correct(tiles, flat, dark)
    t = np.clip(tiles.astype(np.float64) - dark, 0, None)
    m1 = t.max()
    u = t / flat
    want = ((u * m1) / u.max()).astype(np.uint16)
    np.testing.assert_array_equal(out, want)
    assert out.max() <= np.floor(m1)
    # chunked evaluation with precomputed maxima (the multi-GPU / CPU-baseline form) is identical
    parts = [ff.flatfield_maxima(tiles[c], flat, dark) for c in range(2)]
    maxima = (max(p[0] for p in parts), max(p[1] for p in parts))
    assert maxima == ff.flatfield_maxima(tiles, flat, dark)
    chunked = np.stack([ff.flatfield_correct(tiles[c], flat, dark, maxima=maxima) for c in range(2)])
    np.testing.assert_array_equal(chunked, out)


FF_CASES = ("arrays", "scalars", "defaults", "integer_dark", "per_channel", "scalar_flat_array_dark")


def _ff_operand(a):
    return float(a) if a.ndim == 0 else a


def test_flatfield_golden_from_reference_source(golden):
    """tests/golden/flatfield.npz = outputs of the reference's own preprocess.py:62-88."""
    g = golden("flatfield")
    for name in FF_CASES:
        got = ff.flatfield_correct(g["tiles"], _ff_operand(g[name + "__flat"]), _ff_operand(g[name + "__dark"]))
        np.testing.assert_array_equal(got, g[name + "__out"], err_msg=name)
    got = ff.flatfield_correct(g["f32_tiles"], g["arrays__flat"][:16, :24], g["arrays__dark"][:16, :24])
    assert got.dtype == np.float32
    np.testing.assert_array_equal(got, g["f32__out"])


def test_flatfield_against_reference_source_when_present(golden):
    """What the reference's flatfield_correct returned (tests/golden/reference_record.npz), and
    the reference itself when it is present."""
    from oracle._refload import reference_flatfield_correct

    want = golden("reference_record")["flatfield"]
    np.testing.assert_array_equal(ff.flatfield_correct(*flatfield_case()), want)
    ref = reference_flatfield_correct(*flatfield_case())
    if ref is not None:
        np.testing.assert_array_equal(ref, want)


# ---- ROI paths against fixtures made with the reference's real utils.py -----------------------
def test_beads_golden(golden, make_pattern_image):
    d = golden("beads")
    c, t, h, w = (int(v) for v in d["image_shape"])
    image = make_pattern_image(c, t, h, w, salt=int(d["image_salt"]))
    length = int(d["roi_length"])
    beads = d["beads"]
    labels, fg, bg = rois.bead_masks(beads, h, w, length)
    np.testing.assert_array_equal(labels, d["labels"])
    np.testing.assert_array_equal(fg, d["fg"])
    np.testing.assert_array_equal(bg, d["bg"])
    x = np.repeat(beads[:, 1:2], t, 1)
    y = np.repeat(beads[:, 0:1], t, 1)
    np.testing.assert_array_equal(rois.gather_rois(image, x, y, length), d["roi"])


def test_chip_golden(golden, make_pattern_image):
    d = golden("chip")
    c, t, h, w = (int(v) for v in d["image_shape"])
    image = make_pattern_image(c, t, h, w, salt=int(d["image_salt"]))
    length = int(d["roi_length"])
    x, y = d["x"].reshape(-1), d["y"].reshape(-1)
    roi = rois.gather_rois(image, np.repeat(x[:, None], t, 1), np.repeat(y[:, None], t, 1), length)
    np.testing.assert_array_equal(roi, d["roi"])
    fg, bg = rois.chip_masks(x, y, d["fg_radius"].reshape(-1), length, int(d["chamber_radius"]),
                             int(d["max_button_radius"]), w, h)
    src = rois.chip_copy_forward(t, [0])
    np.testing.assert_array_equal(src, np.zeros(t, dtype=np.int64))
    for ti in range(t):
        np.testing.assert_array_equal(fg, d["fg"][:, ti])
        np.testing.assert_array_equal(bg, d["bg"][:, ti])


def chip_multi_inputs(d):
    """(x, y, fg_radius) per search timestep of tests/golden/chip_multi.npz, row-major markers."""
    search = [int(v) for v in d["search_timesteps"]]
    m = d["x"].shape[0]
    refine = d["refine"].reshape(len(search), m, 3)
    radius = np.where(refine[..., 2] >= 0, refine[..., 2], int(d["max_button_radius"]))
    return search, radius


def test_chip_multi_search_golden(golden, make_pattern_image):
    """chip_multi.npz is the output of the reference's own ButtonFinder.__call__ (two search
    timesteps, refinement hits and misses, copy-forward before / between / after them)."""
    d = golden("chip_multi")
    c, t, h, w = (int(v) for v in d["image_shape"])
    image = make_pattern_image(c, t, h, w, salt=int(d["image_salt"]))
    length = int(d["roi_length"])
    search, radius = chip_multi_inputs(d)
    src = rois.chip_copy_forward(t, search)
    np.testing.assert_array_equal(src, [1, 1, 1, 3, 3])
    for ti in range(t):   # copy-forward of centres, find.py:143-151
        np.testing.assert_array_equal(d["x"][:, ti], d["x"][:, src[ti]])
        np.testing.assert_array_equal(d["y"][:, ti], d["y"][:, src[ti]])
    np.testing.assert_array_equal(rois.gather_rois(image, d["x"], d["y"], length), d["roi"])
    for k, ts in enumerate(search):
        fg, bg = rois.chip_masks(d["x"][:, ts], d["y"][:, ts], radius[k], length, int(d["chamber_radius"]),
                                 int(d["max_button_radius"]), w, h)
        for ti in np.nonzero(src == ts)[0]:
            np.testing.assert_array_equal(fg, d["fg"][:, ti])
            np.testing.assert_array_equal(bg, d["bg"][:, ti])


def test_finders_against_reference_source_when_present(golden, make_pattern_image):
    """The committed bead / chip fixtures equal what the reference's own BeadFinder /
    ButtonFinder `__call__` (find.py, executed in place with the stochastic centre finder
    pinned) produce on the same inputs; without the reference, what the oracle's masks and crops
    produce from the same centres."""
    from oracle._refload import reference_bead_finder, reference_button_finder

    d = golden("beads")
    c, t, h, w = (int(v) for v in d["image_shape"])
    image = make_pattern_image(c, t, h, w, salt=int(d["image_salt"]))
    ref = reference_bead_finder(image, ["a", "b"], d["beads"], int(d["roi_length"]))
    if ref is None:   # without the reference: the oracle's restatement of the finders against the same fixtures
        labels, fg, bg = rois.bead_masks(d["beads"], h, w, int(d["roi_length"]))
        x, y = np.repeat(d["beads"][:, 1:2], t, 1), np.repeat(d["beads"][:, 0:1], t, 1)
        ref = {"roi": rois.gather_rois(image, x, y, int(d["roi_length"])), "fg": np.repeat(fg[:, None], t, 1),
               "bg": np.repeat(bg[:, None], t, 1)}
    np.testing.assert_array_equal(ref["roi"], d["roi"])
    for ti in range(t):
        np.testing.assert_array_equal(ref["fg"][:, ti], d["fg"])
        np.testing.assert_array_equal(ref["bg"][:, ti], d["bg"])

    d = golden("chip")
    c, t, h, w = (int(v) for v in d["image_shape"])
    image = make_pattern_image(c, t, h, w, salt=int(d["image_salt"]))
    rows, cols = d["x"].shape
    refine = [None if r[2] < 0 else tuple(int(v) for v in r) for r in d["refine"].reshape(-1, 3)]
    ref = reference_button_finder(image, ["a", "b"], np.full((rows, cols), "default"), d["coarse_x"], d["coarse_y"], refine)
    if ref is None:
        x, y, length = d["x"].reshape(-1), d["y"].reshape(-1), int(d["roi_length"])
        fg, bg = rois.chip_masks(x, y, d["fg_radius"].reshape(-1), length, int(d["chamber_radius"]),
                                 int(d["max_button_radius"]), w, h)
        ref = {"roi": rois.gather_rois(image, np.repeat(x[:, None], t, 1), np.repeat(y[:, None], t, 1), length),
               "fg": np.repeat(fg[:, None], t, 1), "bg": np.repeat(bg[:, None], t, 1), "x": x[:, None]}
    np.testing.assert_array_equal(ref["roi"], d["roi"])
    np.testing.assert_array_equal(ref["fg"], d["fg"])
    np.testing.assert_array_equal(ref["bg"], d["bg"])
    np.testing.assert_array_equal(ref["x"][:, 0], d["x"].reshape(-1))


def test_copy_forward_sources():
    np.testing.assert_array_equal(rois.chip_copy_forward(6, [2, 4]), [2, 2, 2, 2, 4, 4])
    np.testing.assert_array_equal(rois.chip_copy_forward(3, 0), [0, 0, 0])


def test_masked_stats_and_median():
    rng = np.random.default_rng(2)
    roi = rng.integers(0, 65535, (3, 2, 2, 10, 10), dtype=np.uint16, endpoint=True)
    fg = rng.random((3, 2, 10, 10)) < 0.3
    bg = ~fg
    fg[1] = False
    s = red.masked_stats(roi, fg, bg)
    assert s.shape == (3, 2, 2, 8)
    assert np.isnan(s[1, :, :, 4]).all() and (s[1, :, :, 0] == 0).all() and np.isnan(s[1, :, :, 6]).all()
    m, c, t = 2, 1, 0
    vals = roi[m, c, t][fg[m, t]]
    assert s[m, c, t, 0] == vals.size and s[m, c, t, 2] == vals.sum() and s[m, c, t, 4] == vals.mean()
    med = red.masked_median(roi, fg)
    assert med[m, c, t] == np.median(vals) and np.isnan(med[1]).all()
    np.testing.assert_array_equal(s[..., 6], med)
    np.testing.assert_array_equal(s[..., 7], red.masked_median(roi, bg))


def filter_cases(g):
    names = [str(v) for v in g["channels"]]
    k = 0
    while f"case{k}__valid" in g:
        search = [str(v) for v in g[f"case{k}__search"]] or None
        mc = int(g[f"case{k}__min_contrast"])
        yield names, search, (None if mc < 0 else mc), g[f"case{k}__valid"]
        k += 1


def test_filter_expression_golden_from_reference_source(golden):
    """tests/golden/filter.npz = the reference's own filter_expression (filter.py:11-37) run in
    place (composition pinned; xarray's where/median restated, see oracle/_refload.py)."""
    g = golden("filter")
    n = 0
    for names, search, mc, want in filter_cases(g):
        idx = list(range(len(names))) if search is None else [names.index(s) for s in search]
        got = red.filter_expression_valid(g["roi"], g["fg"], g["bg"], g["valid"], idx, mc)
        np.testing.assert_array_equal(got, want)
        n += 1
    assert n == 6


def test_filter_expression_against_reference_source_when_present(golden):
    """filter.npz against the reference's own filter_expression, with xarray's `where` promoting
    to the input type and to float64; without the reference, the oracle against the same golden."""
    from oracle._refload import reference_filter_expression

    g = golden("filter")
    for names, search, mc, want in filter_cases(g):
        idx = list(range(len(names))) if search is None else [names.index(s) for s in search]
        np.testing.assert_array_equal(red.filter_expression_valid(g["roi"], g["fg"], g["bg"], g["valid"], idx, mc), want)
        for promote in (None, np.float64):
            got = reference_filter_expression(g["roi"], g["fg"], g["bg"], g["valid"], names, search, mc, promote)
            if got is not None:
                np.testing.assert_array_equal(got, want)


def test_mrbles_intensities_golden_from_reference_expression(golden):
    """identify.py:76-80 executed in place: bit-identical to the oracle when xarray's `where`
    promotes u16 to float64; within float32 rounding of the MEAN (<= 1e-5 relative to it, the
    north_star tolerance) when it promotes to float32 (xarray.core.dtypes.maybe_promote)."""
    g = golden("filter")
    names = [str(v) for v in g["channels"]]
    idx = [names.index(str(c)) for c in g["intensity_channels"]]
    got = red.mrbles_intensities(g["roi"][:, idx], g["fg"], g["bg"])
    np.testing.assert_array_equal(got, g["intensities_f64"])
    assert np.isnan(got[7]).all()                       # empty foreground
    mean_scale = float(np.nanmax(red.masked_stats(g["roi"][:, idx, :1], g["fg"][:, :1], g["bg"][:, :1])[..., 4]))
    np.testing.assert_allclose(got, g["intensities_f32"], rtol=0, atol=1e-5 * mean_scale)


def test_filter_leaky_golden_from_reference_source(golden):
    """filter.py:65-94 (`filter_leaky_buttons`) executed in place -> leaky* entries of filter.npz."""
    from oracle._refload import reference_filter_leaky

    g = golden("filter")
    names = [str(v) for v in g["channels"]]
    for k in range(3):
        search = [str(v) for v in g[f"leaky{k}__search"]] or None
        idx = list(range(len(names))) if search is None else [names.index(s) for s in search]
        got = red.filter_leaky_valid(g["roi"], g["fg"], g["bg"], g["valid"], g["tag"], g["mark_row"], idx)
        np.testing.assert_array_equal(got, g[f"leaky{k}__valid"])
        ref = reference_filter_leaky(g["roi"], g["fg"], g["bg"], g["valid"], names, g["tag"], g["mark_row"], search)
        if ref is not None:   # build container: the reference's own function again
            np.testing.assert_array_equal(ref, g[f"leaky{k}__valid"])


def test_filter_nonround_golden_from_reference_source(golden):
    """filter.py:40-62 executed in place with the real OpenCV -> tests/golden/nonround.npz."""
    pytest.importorskip("cv2")
    from oracle._refload import reference_filter_nonround

    g = golden("nonround")
    for k in range(3):
        mr = float(g[f"case{k}__min_roundness"])
        np.testing.assert_array_equal(red.filter_nonround_valid(g["fg"], g["valid"], mr), g[f"case{k}__valid"])
        ref = reference_filter_nonround(g["fg"], g["valid"], ["a", "b"], mr)
        if ref is not None:
            np.testing.assert_array_equal(ref, g[f"case{k}__valid"])
