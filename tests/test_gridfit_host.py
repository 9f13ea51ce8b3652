"""magnify_b200/gridfit.py (all comb offsets evaluated at once, closed-form line fits) side by side
with what the reference's own helpers (find.py:630-757) and the tail of ButtonFinder.find_centers
(find.py:233-306) returned on the same inputs (tests/golden/reference_record.npz; the reference
itself too, when it is present): identical labels, fits equal to rounding."""
import numpy as np

from magnify_b200 import gridfit


def reference_find():
    from oracle._refload import load_reference_find

    return load_reference_find()


def jittered_grid(rng, rows, cols, row_dist, col_dist, top, left, drop=0.1, extra=5, shear=0.01):
    yy, xx = np.mgrid[0:rows, 0:cols].astype(float)
    y = top + yy * row_dist + shear * xx * col_dist + rng.normal(0, 1.5, yy.shape)
    x = left + xx * col_dist - shear * yy * row_dist + rng.normal(0, 1.5, yy.shape)
    pts = np.stack([y.ravel(), x.ravel()], 1)
    pts = pts[rng.random(len(pts)) > drop]
    noise = np.stack([rng.uniform(0, top + rows * row_dist + 40, extra), rng.uniform(0, left + cols * col_dist + 40, extra)], 1)
    return np.concatenate([pts, noise])


def helper_cases():
    rng = np.random.default_rng(0)
    for trial in range(12):
        rows, cols = int(rng.integers(2, 9)), int(rng.integers(2, 7))
        row_dist, col_dist = float(rng.uniform(30, 60)), float(rng.uniform(50, 90))
        top, left = float(rng.uniform(10, 60)), float(rng.uniform(10, 60))
        pts = jittered_grid(rng, rows, cols, row_dist, col_dist, top, left)
        shape = (int(top + rows * row_dist + 80), int(left + cols * col_dist + 80))
        yield pts, shape, rows, cols, row_dist, col_dist, left, np.full(rows, cols)


ONE_FIT = (np.array([1.0, 2.0, 4.0]), np.array([2.0, 4.1, 8.2]), np.zeros(3, int), 1, np.array([3]))

ROWS, COLS, ROW_DIST, COL_DIST, SHAPE, CHAMBER_RADIUS = 6, 4, 50.0, 80.0, (400, 420), 20   # chamber_diameter 40
CORNERS = ((None, None), (15, 20))


def centers_case():
    rng = np.random.default_rng(3)
    tag = np.full((ROWS, COLS), "a", dtype="<U8")
    tag[2, 1] = ""
    per_channel = [jittered_grid(rng, ROWS, COLS, ROW_DIST, COL_DIST, 40, 50) for _ in range(2)]
    return tag, per_channel


def grid_centers(tag, per_channel, top, left):
    pts = np.empty((0, 2))
    for new in per_channel:
        pts = gridfit.merge_channel_points(pts, new, CHAMBER_RADIUS)
    return gridfit.grid_centers(pts, tag, SHAPE, ROW_DIST, COL_DIST, CHAMBER_RADIUS, top, left, 10)


def record():
    """This package's side of every comparison with the reference in this module (written to
    tests/golden/reference_record.npz by tests/golden/make_reference_record.py)."""
    out = {}
    for k, (pts, shape, rows, cols, row_dist, col_dist, left, ideal_r) in enumerate(helper_cases()):
        a = gridfit.comb_labels(pts[:, 0], shape[0], rows, row_dist, ideal_r, 10)
        b = gridfit.spaced_labels(pts[:, 1], left - 20, cols, 40, col_dist - 40)
        keep = (a >= 0) & (b >= 0)
        out[f"comb_{k}"], out[f"spaced_{k}"] = a, b
        out[f"fit_slope_{k}"], out[f"fit_icept_{k}"] = gridfit.fit_lines(pts[keep, 1], pts[keep, 0], a[keep], rows, ideal_r)
    out["fit_one"] = np.asarray(gridfit.fit_lines(*ONE_FIT))
    tag, per_channel = centers_case()
    for k, (top, left) in enumerate(CORNERS):
        out[f"centers_x_{k}"], out[f"centers_y_{k}"] = grid_centers(tag, per_channel, top, left)
    return out


def test_helpers_match_reference_functions(golden):
    rec, ref = golden("reference_record"), reference_find()
    for k, (pts, shape, rows, cols, row_dist, col_dist, left, ideal_r) in enumerate(helper_cases()):
        sides = [(gridfit.comb_labels, gridfit.spaced_labels, gridfit.fit_lines)]
        if ref is not None:
            sides.append((ref.cluster_1d, ref.label_clusters, ref.regress_clusters))
        for comb, spaced, fit in sides:
            a = comb(pts[:, 0], shape[0], rows, row_dist, ideal_r, 10)
            np.testing.assert_array_equal(a, rec[f"comb_{k}"])
            b = spaced(pts[:, 1], left - 20, cols, 40, col_dist - 40)
            np.testing.assert_array_equal(b, rec[f"spaced_{k}"])
            keep = (a >= 0) & (b >= 0)
            got = fit(pts[keep, 1], pts[keep, 0], a[keep], rows, ideal_r)
            np.testing.assert_allclose(got[0], rec[f"fit_slope_{k}"], rtol=1e-10)
            np.testing.assert_allclose(got[1], rec[f"fit_icept_{k}"], rtol=1e-10, atol=1e-9)
    np.testing.assert_allclose(gridfit.fit_lines(*ONE_FIT), rec["fit_one"], rtol=1e-12)
    if ref is not None:
        np.testing.assert_allclose(ref.regress_clusters(*ONE_FIT), rec["fit_one"], rtol=1e-12)


def test_grid_centers_matches_reference_find_centers_tail(golden, monkeypatch):
    """ButtonFinder.find_centers with its circle finder pinned to given points
    (find.py:205-306) == gridfit.merge_channel_points + grid_centers."""
    rec, ref = golden("reference_record"), reference_find()
    tag, per_channel = centers_case()
    for k, (top, left) in enumerate(CORNERS):
        got_x, got_y = grid_centers(tag, per_channel, top, left)
        np.testing.assert_allclose(got_x, rec[f"centers_x_{k}"], rtol=1e-10, atol=1e-8)
        np.testing.assert_allclose(got_y, rec[f"centers_y_{k}"], rtol=1e-10, atol=1e-8)
        if ref is None:
            continue
        want_x, want_y = reference_find_centers(ref, monkeypatch, tag, per_channel, top, left)
        np.testing.assert_allclose(want_x, rec[f"centers_x_{k}"], rtol=1e-10, atol=1e-8)
        np.testing.assert_allclose(want_y, rec[f"centers_y_{k}"], rtol=1e-10, atol=1e-8)


def reference_find_centers(ref, monkeypatch, tag, per_channel, top, left):
    """The reference's ButtonFinder.find_centers executed in place on points pinned per channel."""
    from oracle._refload import LabelledArray

    class Counts:
        def __init__(self, mask):
            self.mask = mask

        def sum(self, dim):
            return LabelledArray(self.mask.sum(axis=1 if dim == "mark_col" else 0), ("k",), {})

    class Tag:
        def __ne__(self, other):
            return Counts(tag != other)

    assay = type("A", (), {"tag": Tag(), "sizes": {"mark_row": ROWS, "mark_col": COLS}})()
    images = [LabelledArray(np.zeros(SHAPE, np.uint8), ("im_y", "im_x"), {}) for _ in per_channel]
    finder = ref.ButtonFinder(row_dist=ROW_DIST, col_dist=COL_DIST, min_button_diameter=10, max_button_diameter=24,
                              chamber_diameter=40, top_chamber=top, left_chamber=left, low_edge_quantile=0.1,
                              high_edge_quantile=0.9, num_iter=100, min_roundness=0.2, cluster_penalty=10,
                              roi_length=None, progress_bar=False, search_timestep=0, search_channel=None,
                              interactive=False)
    assert finder.chamber_radius == CHAMBER_RADIUS
    calls = iter(per_channel)

    def pinned_circles(img, **kw):
        pts = next(calls)
        return np.column_stack([pts, np.full(len(pts), 9.0)]), None

    monkeypatch.setattr(ref.utils, "find_circles", pinned_circles)
    return finder.find_centers(images, assay)
