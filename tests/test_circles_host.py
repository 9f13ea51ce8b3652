"""Host formulas of the circle finder front end (magnify_b200/circles.py) against NumPy itself,
and the cv2/NumPy oracle against what the reference's own find_circles stages returned
(tests/golden/reference_record.npz; the reference itself too, when it is present)."""
import numpy as np
import pytest

from magnify_b200 import circles as mc


def synthetic_discs(h, w, discs, seed=0, noise=12, level=3000, dtype=np.uint16):
    rng = np.random.default_rng(seed)
    img = (rng.random((h, w)) * noise).astype(np.float64) * 20
    yy, xx = np.mgrid[0:h, 0:w]
    for cy, cx, r in discs:
        img[(yy - cy) ** 2 + (xx - cx) ** 2 <= r * r] += level
    return img.astype(dtype)


def test_linear_quantile_is_numpy_quantile():
    rng = np.random.default_rng(0)
    for trial in range(1500):
        n = int(rng.integers(1, 5000)) if trial % 3 else int(rng.integers(1, 40))
        a = np.sqrt(rng.integers(0, 33_000_000, n).astype(np.float32)) if trial % 2 else \
            rng.integers(0, 50, n).astype(np.float32)
        q = float(rng.random()) if trial % 5 else [0.0, 1.0, 0.5, 0.1, 0.9][trial % 7 % 5]
        if trial % 11 == 0:
            q = np.float64(1 - np.pi * 8 / 72**2)          # the chip finder's high quantile, find.py:345-347
        want = np.quantile(a, q)
        srt = np.sort(a)
        _, prev, nxt = mc._quantile_indexes(n, q)
        lower = srt[prev]
        upper = srt[min(nxt, n - 1)] if prev != -1 else srt[-1]
        got = mc.linear_quantile(n, q, lower, upper, srt[-1])
        assert got == want and got.dtype == want.dtype, (n, q, got, want)
    with pytest.raises(ValueError):
        mc._quantile_indexes(10, 1.5)


def test_canny_thresholds():
    assert mc.canny_thresholds(3.5, 10.25) == (12, 105)
    assert mc.canny_thresholds(10.25, 3.5) == (12, 105)            # swapped when out of order
    assert mc.canny_thresholds(0.0, 40000.0) == (0, 32767 * 32767)
    assert mc.canny_thresholds(-2.0, 2.0) == (-2, 4)


EDGE_QUANTILES = ((0.1, 0.9), (0.5, 0.97))


def edge_image():
    from oracle import circles as oc

    return oc.to_uint8(synthetic_discs(300, 260, [(60, 70, 15), (150, 120, 22), (220, 200, 12), (100, 200, 18)]))


def to_uint8_inputs():
    return [synthetic_discs(20, 30, [(10, 10, 5)]), np.full((4, 4), 7, np.uint16), np.zeros((0, 3), np.float32),
            synthetic_discs(20, 30, [(10, 10, 5)], dtype=np.float32) - 50]


PERIMETER_RADII = list(range(1, 40)) + [60, 100, 255]


def neighbor_cases():
    rng = np.random.default_rng(0)
    for trial in range(120):
        n, min_dist = int(rng.integers(1, 300)), int(rng.integers(1, 12))
        c = np.stack([rng.integers(-5, 120, n), rng.integers(-5, 150, n), rng.integers(3, 20, n)], 1).astype(np.int32)
        if trial % 3 == 0:
            c[:, :2] = np.abs(c[:, :2])
        yield c, min_dist


def circumcircle_cases():
    """Three edge pixels in one grid cell per trial."""
    rng = np.random.default_rng(0)
    for trial in range(25):
        pts = set()
        while len(pts) < 3:
            pts.add((int(rng.integers(20, 40)), int(rng.integers(40, 60))))
        yield sorted(pts)


def circle_set(rows):
    return {tuple(row.view(np.uint32).tolist()) for row in np.asarray(rows, np.float32).reshape(-1, 3)}


def grid_case():
    """Edge stages of a small disc image and circles sampled from its grid lists."""
    from oracle import circles as oc

    img = oc.to_uint8(synthetic_discs(120, 150, [(40, 50, 14), (80, 100, 20), (30, 120, 9)], noise=6))
    st = oc.edge_stages(img, 0.3, 0.95)
    rng = np.random.default_rng(1)
    raw = oc.sampled_circles(st["edges"], 20, rng.integers(0, 2**32, (400, 3), dtype=np.uint64))
    return img, st, oc.filter_round(raw, 6, 24, img.shape)


def record():
    """This package's side of every comparison with the reference in this module (written to
    tests/golden/reference_record.npz by tests/golden/make_reference_record.py)."""
    from oracle import circles as oc

    out = {}
    img = edge_image()
    for k, (low_q, high_q) in enumerate(EDGE_QUANTILES):
        out[f"edges{k}"] = oc.edge_stages(img, low_q, high_q)["edges"]
    for k, arr in enumerate(to_uint8_inputs()):
        out[f"to_uint8_{k}"] = oc.to_uint8(arr)
    for r in PERIMETER_RADII:
        for four in (False, True):
            out[f"perimeter_{r}_{int(four)}"] = mc.circle_perimeter(r, four)
    for k, (c, min_dist) in enumerate(neighbor_cases()):
        out[f"neighbors_{k}"] = mc.filter_neighbors(c, min_dist)
    for k, pts in enumerate(circumcircle_cases()):
        out[f"circumcircles_{k}"] = np.array(sorted(circle_set([oc.circumcircle(a, b, c) for a in pts for b in pts
                                                                 for c in pts])), np.uint32).view(np.float32)
    _, st, circles = grid_case()
    out["grid_coords"], out["grid_starts"], out["grid_counts"] = oc.grid_lists(st["edges"], 20)
    out["grid_scores"] = oc.perimeter_scores(circles, st["edges"], st["dx"], st["dy"], 24)
    return out


def test_oracle_edges_are_the_reference_functions_edges(golden):
    """tests/golden/reference_record.npz holds the edges and uint8 conversions the reference's
    own find_circles stages and utils.to_uint8 returned; checked against the reference itself
    when it is present."""
    from oracle import circles as oc
    from oracle._refload import load_reference_utils, reference_find_circles_stages

    pytest.importorskip("cv2")
    rec = golden("reference_record")
    img = edge_image()
    for k, (low_q, high_q) in enumerate(EDGE_QUANTILES):
        np.testing.assert_array_equal(oc.edge_stages(img, low_q, high_q)["edges"], rec[f"edges{k}"])
        ref = reference_find_circles_stages(img, low_q, high_q, 20, 2000, 8, 30, 0.2, 8)
        if ref is not None:
            np.testing.assert_array_equal(ref[0], rec[f"edges{k}"])
    utils = load_reference_utils()
    for k, arr in enumerate(to_uint8_inputs()):
        np.testing.assert_array_equal(oc.to_uint8(arr), rec[f"to_uint8_{k}"])
        if utils is not None:
            np.testing.assert_array_equal(utils.to_uint8(arr), rec[f"to_uint8_{k}"])


def test_perimeter_and_suppression_match_reference_numba(golden):
    """circle_points and filter_neighbors as the reference's numba functions returned them."""
    from oracle._refload import load_reference_utils

    rec, utils = golden("reference_record"), load_reference_utils()
    for r in PERIMETER_RADII:
        for four in (False, True):
            want = rec[f"perimeter_{r}_{int(four)}"]
            np.testing.assert_array_equal(mc.circle_perimeter(r, four), want)
            if utils is not None:
                np.testing.assert_array_equal(utils.circle_points(r, four), want)
    for k, (c, min_dist) in enumerate(neighbor_cases()):
        np.testing.assert_array_equal(mc.filter_neighbors(c, min_dist), rec[f"neighbors_{k}"])
        if utils is not None:
            np.testing.assert_array_equal(utils.filter_neighbors(c, min_dist), rec[f"neighbors_{k}"])
    assert mc.filter_neighbors(np.empty((0, 3), np.int32), 3).shape == (0,)


def test_oracle_circumcircle_is_numbas_arithmetic(golden):
    """Three edge pixels in one grid cell: the reference's candidate_circles can only produce the
    27 ordered draws of them, so the SET of its float32 outputs pins the arithmetic bit for bit."""
    from oracle import circles as oc
    from oracle._refload import load_reference_utils

    rec, utils = golden("reference_record"), load_reference_utils()
    for trial, pts in enumerate(circumcircle_cases()):
        want = circle_set(rec[f"circumcircles_{trial}"])
        assert circle_set([oc.circumcircle(a, b, c) for a in pts for b in pts for c in pts]) == want, trial
        if utils is not None:
            edges = np.zeros((100, 100), np.uint8)
            for r, c in pts:
                edges[r, c] = 1
            assert circle_set(utils.candidate_circles(edges, 20, 3000)) == want, trial


def test_oracle_grid_lists_and_scores_match_reference_numba(golden):
    from oracle import circles as oc
    from oracle._refload import load_reference_utils

    rec, utils = golden("reference_record"), load_reference_utils()
    img, st, circles = grid_case()
    assert len(circles) > 20
    coords, starts, counts = oc.grid_lists(st["edges"], 20)
    np.testing.assert_array_equal(coords, rec["grid_coords"])
    np.testing.assert_array_equal(starts, rec["grid_starts"])
    np.testing.assert_array_equal(counts, rec["grid_counts"])
    mine = oc.perimeter_scores(circles, st["edges"], st["dx"], st["dy"], 24)
    np.testing.assert_array_equal(mine, rec["grid_scores"])
    if utils is None:
        return
    rc, rs, rn = utils.grid_array(st["edges"], 20)
    np.testing.assert_array_equal(rc, rec["grid_coords"])
    np.testing.assert_array_equal(rs, rec["grid_starts"])
    np.testing.assert_array_equal(rn, rec["grid_counts"])
    # scores: the reference's own mean_grad on the same circles
    pad = 2 * 24
    angles, padded = np.pad(np.arctan2(st["dy"], st["dx"]), pad), np.pad(st["edges"], pad)
    for k, (row, col, radius) in enumerate(circles):
        pts = utils.circle_points(int(radius))
        want = utils.mean_grad(angles, padded, np.array([[row + pad, col + pad]], np.int32), pts)[0] / len(pts)
        assert rec["grid_scores"][k] == np.float32(want), (k, rec["grid_scores"][k], want)
