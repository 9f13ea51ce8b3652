"""The drop-in claim, executed: the reference's own UNMODIFIED package (registry.py, pipeline.py,
preprocess.py, stitch.py, find.py, identify.py, postprocess.py, reader.py ...) is imported in
place (oracle/_refload.py::load_reference_package), `magnify_b200.components.install()` replaces
its hot-path components in its own registry, and the reference's own builders
(`microfluidic_chip_pipe`, `beads_pipe`, `mrbles_pipe`, `mg.microfluidic_chip`, `mg.beads`, `mg.mrbles`;
registry.py:32-612)
run `Pipeline.__call__` (pipeline.py:14-29) over them.  The resulting dataset must be IDENTICAL
(variables, dims, dtypes, coordinates, attrs, values) to the one the reference's own components
produce through the same pipe on the same input.

This container has the reference but no GPU, so the array kernels under the components are
stood in for by the oracle (tests/cpu_ops.py); the same component layer runs on the real
kernels in tests/test_gpu_dropin.py against goldens written by this file's generator
(tests/golden/make_dropin_golden.py).  The stochastic circle search of the reference
(`utils.find_circles`, unseeded; SURVEY.md section 0 fact 4) is pinned on BOTH sides to one
deterministic detector, so the centres, the grid fit (find.py:233-306 vs magnify_b200.gridfit)
and the per-chamber refinement (find.py:336-378 vs ButtonFinder.refine) are compared too.
"""
import numpy as np
import pytest

from dropin_cases import (assert_same_dataset, bead_input, chip_input, deterministic_find_circles, draw_chip, installed,
                          load_mg, mrbles_input, pin_circle_finders, replay_bead_case, replay_chip_case)


@pytest.fixture()
def mg_or_none(monkeypatch):
    mod = load_mg()
    if mod is not None:
        pin_circle_finders(monkeypatch, mod)
    return mod


@pytest.fixture()
def mg(mg_or_none):
    if mg_or_none is None:
        pytest.skip("the reference package is not present")
    return mg_or_none


def test_registry_and_pipeline_surface(mg, monkeypatch):
    """install() registers under the reference's names; the reference's builders then resolve to
    the GPU factories, with the reference's own kwargs (registry.py:243-269, 431-449, 593-610)."""
    from magnify_b200 import components

    with installed(mg, monkeypatch) as names:
        assert {"stitch", "stitch_b200", "flatfield_correct", "find_buttons", "find_beads", "quantify"} <= set(names)
        reg = mg.registry.components
        assert reg.get("stitch") is components.make_stitch
        assert reg.get("find_buttons") is components.make_find_buttons
        pipe = mg.microfluidic_chip_pipe(shape=(2, 2), overlap=0, chip_type="pc", search_channel="a")
        order = [name for name, _ in pipe.components]
        assert order == ["standardize_format", "identify_buttons", "stitch", "rotate", "find_buttons", "drop",
                         "restore_format"]
        comps = dict(pipe.components)
        assert isinstance(comps["stitch"], components.Stitcher) and comps["stitch"].overlap == 0
        finder = comps["find_buttons"]
        assert isinstance(finder, components.ButtonFinder)
        assert (finder.row_dist, finder.col_dist) == (406 / 3.22, 750 / 3.22)          # chip_type="pc"
        pipe = mg.beads_pipe(flatfield=1.25, darkfield=3.0, min_bead_diameter=6, max_bead_diameter=20)
        comps = dict(pipe.components)
        assert isinstance(comps["find_beads"], components.BeadFinder) and comps["find_beads"].roi_length == 40
        # add_pipe / remove_pipe (pipeline.py:31-87) with the additive component
        pipe.add_pipe("quantify", after="find_beads")
        assert [n for n, _ in pipe.components][3:5] == ["find_beads", "quantify"]
        with pytest.raises(ValueError):
            pipe.add_pipe("quantify")                     # names are unique in a pipe
        pipe.remove_pipe("quantify")
        with pytest.raises(ValueError):
            mg.registry.components.get("find_buttons")(1, 1, 30, 20, 60, *([None] * 12))   # min > max diameter
    assert mg.registry.components.get("stitch") is not components.make_stitch           # restored


@pytest.mark.parametrize("case", ["chip_single", "chip_series", "chip_tiles", "chip_blank_float"])
def test_chip_pipeline_identical_to_reference(mg_or_none, monkeypatch, case):
    """Without the reference: the component layer on the CPU stand-in replays the reference's
    pipeline states recorded in tests/golden/dropin_<case>.npz."""
    mg = mg_or_none
    if mg is None:
        import cpu_ops

        cpu_ops.patch_components(monkeypatch)
        replay_chip_case(case, on_device=False)
        return
    data, kwargs = chip_input(case)
    want = mg.microfluidic_chip(data, **kwargs)
    with installed(mg, monkeypatch):
        got = mg.microfluidic_chip(data, **kwargs)
    assert_same_dataset(got, want)


@pytest.mark.parametrize("case", ["beads_single", "beads_flatfield_tiles", "beads_none"])
def test_beads_pipeline_identical_to_reference(mg_or_none, monkeypatch, case):
    mg = mg_or_none
    if mg is None:
        import cpu_ops

        cpu_ops.patch_components(monkeypatch)
        replay_bead_case(case)
        return
    data, kwargs = bead_input(case)
    want = mg.beads(data, **kwargs)
    with installed(mg, monkeypatch):
        got = mg.beads(data, **kwargs)
    assert_same_dataset(got, want)


def test_mrbles_pipeline_identical_to_reference(mg, monkeypatch, tmp_path):
    """`mg.mrbles` (registry.py:272-449): flatfield_correct -> stitch -> find_beads from this package,
    then the reference's OWN identify_mrbles (identify.py:49-232: `where(fg).mean - where(bg).median`
    intensities, lanthanide volumes by least squares, code assignment by the mixture model) consumes
    their output.  Volumes, ratios and the code of every bead must come out as through the
    reference's own components."""
    data, kwargs = mrbles_input(str(tmp_path))
    want = mg.mrbles(data, **kwargs)
    with installed(mg, monkeypatch):
        pipe = mg.mrbles_pipe(**{k: v for k, v in kwargs.items()})
        assert [n for n, _ in pipe.components] == ["standardize_format", "flatfield_correct", "stitch", "find_beads",
                                                   "identify_mrbles", "drop", "restore_format"]
        got = mg.mrbles(data, **kwargs)
    assert_same_dataset(got, want)
    tags = np.asarray(want["tag"].values)
    assert len(tags) == 24 and {"code_a", "code_b", "code_c"} <= set(tags.tolist())     # the fixture really separates the codes
    assert np.isfinite(np.asarray(want["ln_ratio"].values)).all()


@pytest.mark.parametrize("case", ["chip_series", "chip_blank_float"])
def test_chip_pipe_with_filters(mg, monkeypatch, case):
    """The consumers of the crops, through the registry: filter_expression, filter_nonround and
    filter_leaky (filter.py:11-94) added to the chip pipe with add_pipe.  install() replaces all
    three (medians and contour perimeters from the kernels); `valid` and everything else must come
    out as from the reference's own filters, on a time series and on a chip with a blank chamber."""
    data, kwargs = chip_input(case)

    def build():
        pipe = mg.microfluidic_chip_pipe(**kwargs)
        pipe.add_pipe("filter_expression", after="find_buttons")
        pipe.add_pipe("filter_nonround", after="filter_expression", min_roundness=0.6)
        pipe.add_pipe("filter_leaky", after="filter_nonround")
        return pipe

    want = build()(data)
    with installed(mg, monkeypatch):
        from magnify_b200 import components

        pipe = build()
        for name in ("filter_expression", "filter_nonround", "filter_leaky"):     # really this package's
            assert dict(pipe.components)[name].__module__ == components.__name__
        got = pipe(data)
    assert_same_dataset(got, want)
    assert np.asarray(want["valid"].values).any()


def test_chip_pipe_with_flatfield_and_quantify(mg, monkeypatch):
    """BASELINE config 3's pipe: the chip pipe has no flat-field step (registry.py:243-269), it is
    inserted with add_pipe (pipeline.py:31-78; SURVEY.md section 0 fact 8).  The lazy
    flatfield_correct + stitch pair must equal the reference's two components, and `quantify`
    must equal the xarray expressions it replaces (identify.py:76-80, README.md:21-22)."""
    data, kwargs = chip_input("chip_series")
    kwargs = {k: v for k, v in kwargs.items()}
    h, w = data.sizes["y"], data.sizes["x"]
    yy, xx = np.mgrid[0:h, 0:w]
    flat = 1.0 + 0.3 * np.sin(yy / 37.0) * np.cos(xx / 51.0)
    dark = 20.0 + 3.0 * np.cos(yy / 29.0)

    def build():
        pipe = mg.microfluidic_chip_pipe(**kwargs)
        pipe.add_pipe("flatfield_correct", after="standardize_format", flatfield=flat, darkfield=dark)
        return pipe

    want = build()(data)
    with installed(mg, monkeypatch):
        pipe = build()
        pipe.add_pipe("quantify", after="find_buttons")
        got = pipe(data)
    extra = ["fg_sum", "bg_sum", "fg_mean", "bg_mean", "fg_count", "bg_count", "fg_median", "bg_median"]
    assert_same_dataset(got.drop_vars(extra), want)
    # the summaries against the reference-side expressions on the reference's dataset
    w2 = want.transpose("mark_row", "mark_col", "channel", "time", "roi_y", "roi_x")
    g2 = got.transpose("mark_row", "mark_col", "channel", "time", "roi_y", "roi_x")
    for mask in ("fg", "bg"):
        sel = w2.roi.where(w2[mask])
        np.testing.assert_allclose(g2[mask + "_mean"].values, sel.mean(dim=["roi_x", "roi_y"]).values, rtol=1e-6)
        np.testing.assert_array_equal(g2[mask + "_median"].values, sel.median(dim=["roi_x", "roi_y"]).values)
        np.testing.assert_array_equal(g2[mask + "_count"].values, w2[mask].sum(dim=["roi_x", "roi_y"]).values)


def test_deterministic_detector_is_a_fair_pin():
    """The pinned detector finds the drawn buttons (so the comparison exercises real geometry).
    oracle.circles.to_uint8 is the reference's utils.to_uint8 (tests/test_circles_host.py)."""
    from oracle import circles as oc

    img = oc.to_uint8(draw_chip((3, 3)))            # the image of chip_input("chip_single")
    circles, scores = deterministic_find_circles(img, min_radius=8, max_radius=16)
    assert len(circles) == 9 and (np.abs(circles[:, 2] - 10) <= 1).all()
