"""The oracle's integer geometry against the golden vectors made from the reference's real
utils.py (tests/golden/make_golden.py and make_reference_record.py), against cv2, and -- when
the reference is present -- against the reference itself."""
import numpy as np
import pytest

from oracle import geometry as g
from oracle._refload import load_reference_utils


def test_bounding_box_golden(golden):
    d = golden("geometry")
    for args, want in zip(d["bb_args"], d["bb_out"]):
        assert g.bounding_box(*[int(v) for v in args]) == tuple(int(v) for v in want)


def test_bounding_box_known_answers():
    # SURVEY.md section 8c, obtained from the reference's utils.bounding_box
    assert g.bounding_box(5, 5, 100, 2048, 2048) == (0, 100, 0, 100)
    assert g.bounding_box(2040, 1000, 100, 2048, 2048) == (950, 1050, 1948, 2048)
    assert g.bounding_box(100, 100, 71, 2048, 2048) == (65, 136, 65, 136)


def test_disc_tables_golden(golden):
    d = golden("geometry")
    hw, area, perim = d["disc_halfwidth"], d["disc_area"], d["perimeter_len"]
    for r in range(1, hw.shape[0]):
        got = g.disc_halfwidths(r)
        np.testing.assert_array_equal(got, hw[r, : r + 1])
        assert len(g.filled_circle_points(r)) == area[r]
        assert len(g.circle_points(r)) == perim[r]
    # areas quoted in SURVEY.md section 7
    assert [int(area[r]) for r in (5, 10, 12, 25)] == [93, 341, 473, 2021]
    with pytest.raises(ValueError):
        g.circle_points(0)


def test_circle_labels_golden(golden):
    d = golden("beads")
    c, t, h, w = (int(v) for v in d["image_shape"])
    labels = g.circle_labels(d["beads"].astype(int), h, w)
    np.testing.assert_array_equal(labels, d["labels"])
    assert set(np.unique(labels)) >= {-2, -1, 0}
    # two r=10 beads 15 px apart (SURVEY.md section 8c): {-2: 58, 0: 283, 1: 283}
    lab = g.circle_labels(np.array([[30, 30, 10], [30, 45, 10]]), 60, 80)
    assert {int(k): int((lab == k).sum()) for k in (-2, 0, 1)} == {-2: 58, 0: 283, 1: 283}


def test_cv_circle_closed_form(golden):
    d = golden("masks_cv")
    for (cy, cx, r, ro, ri), disc, ring in zip(d["cases"], d["disc"], d["ring"]):
        np.testing.assert_array_equal(g.circle((72, 72), (cy, cx), r), disc)
        np.testing.assert_array_equal(g.annulus((72, 72), (cy, cx), ro, ri), ring)
    assert g.circle((72, 72), (36, 36), 10).sum() == 317
    assert g.annulus((72, 72), (36, 36), 30, 16).sum() == 2024


def test_cv_circle_against_cv2():
    cv = pytest.importorskip("cv2")
    for r in list(range(0, 40)) + [64, 100, 200, 256]:
        for cy, cx in [(36, 36), (0, 0), (71, 71), (-4, 20), (30, 80), (5, 66)]:
            img = np.zeros((72, 72), np.uint8)
            cv.circle(img, (cx, cy), r, 1, thickness=-1)
            np.testing.assert_array_equal(g.circle((72, 72), (cy, cx), r), img.astype(bool))


GEOMETRY_RADII = (1, 2, 3, 7, 16, 33, 100, 257)


def geometry_cases():
    rng = np.random.default_rng(0)
    boxes = []
    for _ in range(3000):
        w, h, length = rng.integers(1, 300, 3)
        x, y = rng.integers(-50, 350, 2)
        boxes.append((int(x), int(y), int(length), int(w), int(h)))
    beads = np.stack([rng.integers(-5, 150, 40), rng.integers(-5, 170, 40), rng.integers(1, 20, 40)], 1)
    return boxes, beads


def sorted_points(points):
    return np.array(sorted(map(tuple, np.asarray(points).tolist())))


def record():
    """This package's side of every comparison with the reference in this module (written to
    tests/golden/reference_record.npz by tests/golden/make_reference_record.py)."""
    boxes, beads = geometry_cases()
    out = {"bounding_boxes": np.array([g.bounding_box(*args) for args in boxes]),
           "circle_labels": g.circle_labels(beads, 140, 160)}
    for r in GEOMETRY_RADII:
        out[f"circle_points_{r}"], out[f"circle_points4_{r}"] = g.circle_points(r), g.circle_points(r, True)
        out[f"filled_circle_points_{r}"] = sorted_points(g.filled_circle_points(r))
    return out


def test_against_reference_utils_when_present(golden):
    """What the reference's utils.py returned (tests/golden/reference_record.npz), and the
    reference itself when it is present."""
    rec, u = golden("reference_record"), load_reference_utils()
    boxes, beads = geometry_cases()
    for args, want in zip(boxes, rec["bounding_boxes"]):
        assert g.bounding_box(*args) == tuple(int(v) for v in want)
        if u is not None:
            assert tuple(int(v) for v in u.bounding_box(*args)) == tuple(int(v) for v in want)
    sides = [g] if u is None else [g, u]
    for r in GEOMETRY_RADII:
        for side in sides:
            np.testing.assert_array_equal(side.circle_points(r), rec[f"circle_points_{r}"])
            np.testing.assert_array_equal(side.circle_points(r, True), rec[f"circle_points4_{r}"])
            np.testing.assert_array_equal(sorted_points(side.filled_circle_points(r)), rec[f"filled_circle_points_{r}"])
    for side in sides:
        np.testing.assert_array_equal(side.circle_labels(beads, 140, 160), rec["circle_labels"])
