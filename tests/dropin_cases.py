"""Shared pieces of the drop-in tests (tests/test_dropin_reference.py, tests/golden/make_dropin_golden.py,
tests/test_gpu_dropin.py): inputs shaped like the reference's own test fixtures
(tests/test_chip.py:9-34 `draw_chip`, tests/test_beads.py:9-36 `draw_beads`), one deterministic
circle detector that pins the reference's unseeded random search on both sides, and the dataset
comparison."""
from __future__ import annotations

import contextlib
import json
import os
import tempfile

import numpy as np


def load_mg():
    from oracle._refload import load_reference_package

    return load_reference_package()


# ---------------------------------------------------------------------------------------------
# deterministic stand-in for utils.find_circles (utils.py:100-218), used by BOTH pipelines
# ---------------------------------------------------------------------------------------------
def deterministic_find_circles(img, low_edge_quantile=0.1, high_edge_quantile=0.9, grid_length=20, num_iter=0,
                               min_radius=1, max_radius=10**6, min_dist=0, min_roundness=0.0, gui=None):
    """Bright blobs of a uint8 image as circles: rows (row, col, radius) int32 sorted by score
    (area) descending, like the reference returns its circles best first."""
    import cv2 as cv

    img = np.asarray(img)
    if img.size == 0 or img.max() == 0:
        return np.empty((0, 3), dtype=np.int32), np.empty(0, dtype=np.float32)
    n, _, stats, centroids = cv.connectedComponentsWithStats((img > 127).astype(np.uint8), connectivity=8)
    rows = []
    for k in range(1, n):
        area = int(stats[k, cv.CC_STAT_AREA])
        r = int(round(np.sqrt(area / np.pi)))
        if min_radius <= r <= max_radius:
            rows.append((area, int(round(centroids[k][1])), int(round(centroids[k][0])), r))
    rows.sort(key=lambda v: (-v[0], v[1], v[2]))
    circles = np.array([[r[1], r[2], r[3]] for r in rows], dtype=np.int32).reshape(-1, 3)
    top = max((r[0] for r in rows), default=1)
    scores = np.array([r[0] / (top + 1.0) for r in rows], dtype=np.float32)
    return circles, scores


def pin_circle_finders(monkeypatch, mg):
    """Both circle finders -> the deterministic detector: the reference's `utils.find_circles`
    and this package's `circles.find_circles` / `circles.to_uint8` (GPU code)."""
    import torch

    from magnify_b200 import circles

    monkeypatch.setattr(mg.utils, "find_circles", deterministic_find_circles)

    def to_uint8(x, batched=False):
        arr = x.detach().cpu().numpy()
        if batched:
            return torch.from_numpy(np.stack([mg.utils.to_uint8(a) for a in arr]) if len(arr) else arr.astype(np.uint8))
        return torch.from_numpy(mg.utils.to_uint8(arr))

    def find_circles(image, low_edge_quantile, high_edge_quantile, grid_length, num_iter, min_radius, max_radius,
                     min_roundness, min_dist, seed=0):
        arr = image.detach().cpu().numpy()
        kw = dict(min_radius=min_radius, max_radius=max_radius)
        if arr.ndim == 3:
            return [deterministic_find_circles(a, **kw) for a in arr]
        return deterministic_find_circles(arr, **kw)

    monkeypatch.setattr(circles, "to_uint8", to_uint8)
    monkeypatch.setattr(circles, "find_circles", find_circles)


@contextlib.contextmanager
def installed(mg, monkeypatch):
    """components.install() into the reference's registry, on the CPU stand-in for the kernels;
    the registry is put back afterwards."""
    import cpu_ops
    from magnify_b200 import components

    reg = mg.registry.components
    saved = dict(reg._items)
    with monkeypatch.context() as mp:
        cpu_ops.patch_components(mp)
        try:
            yield components.install()
        finally:
            reg._items = saved


# ---------------------------------------------------------------------------------------------
# inputs
# ---------------------------------------------------------------------------------------------
def _disc(r):
    yy, xx = np.mgrid[-r:r + 1, -r:r + 1]
    return np.argwhere(yy * yy + xx * xx <= r * r) - r


def draw_chip(shape, button_diameter=20, row_dist=100, col_dist=100, value=1000, blanks=(), dtype=np.uint16, jitter=None):
    r = button_diameter // 2
    chip = np.zeros(((shape[0] + 1) * row_dist, (shape[1] + 1) * col_dist), dtype=dtype)
    pts = _disc(r)
    for i in range(shape[0]):
        for j in range(shape[1]):
            if (i, j) in set(blanks):
                continue
            dy, dx = (0, 0) if jitter is None else jitter[i, j]
            chip[pts[:, 0] + (i + 1) * row_dist + dy, pts[:, 1] + (j + 1) * col_dist + dx] = value
    return chip


def _noise(shape, seed, scale=40):
    return np.random.default_rng(seed).integers(0, scale, shape)


def _split_tiles(image, rows, cols, overlap):
    """Cut an image into rows x cols tiles that stitch back to it with `overlap` (stitch.py:22-39):
    every tile carries overlap//2 extra pixels (+ the odd one at the bottom / right) around its part."""
    h, w = image.shape[-2] // rows, image.shape[-1] // cols
    clip, rem = overlap // 2, overlap % 2
    pad = np.pad(image, [(0, 0)] * (image.ndim - 2) + [(clip, clip + rem), (clip, clip + rem)], mode="reflect")
    tiles = np.empty(image.shape[:-2] + (rows, cols, h + overlap, w + overlap), dtype=image.dtype)
    for i in range(rows):
        for j in range(cols):
            tiles[..., i, j, :, :] = pad[..., i * h:i * h + h + overlap, j * w:j * w + w + overlap]
    return tiles


def chip_input(case):
    """(DataArray, kwargs of mg.microfluidic_chip) for a named case."""
    import xarray as xr

    base = dict(min_button_diameter=16, max_button_diameter=32, overlap=0, row_dist=100, col_dist=100, num_iter=1000)
    rng = np.random.default_rng(7)
    if case == "chip_single":
        data = xr.DataArray(data=draw_chip((3, 3)), dims=("y", "x"))
        return data, dict(base, shape=(3, 3))
    if case == "chip_series":
        jit = rng.integers(-6, 7, (3, 4, 2))
        frames = []
        for ch, amp in (("a", 1000), ("b", 400)):
            frames.append([draw_chip((3, 4), value=int(amp * (1 + 0.2 * t)), jitter=jit) + _noise((400, 500), 10 * t + amp)
                           for t in range(3)])
        arr = np.asarray(frames, dtype=np.uint16)
        data = xr.DataArray(data=arr, dims=("channel", "time", "y", "x"),
                            coords={"channel": ["a", "b"], "time": [0, 10, 20]})
        return data, dict(base, shape=(3, 4), search_channel="a", search_timestep=[1])
    if case == "chip_tiles":
        chip = draw_chip((3, 3)) + _noise((400, 400), 3).astype(np.uint16)
        tiles = _split_tiles(chip, 2, 2, 11)
        data = xr.DataArray(data=tiles, dims=("row", "col", "y", "x"))
        return data, dict(base, shape=(3, 3), overlap=11)
    if case == "chip_blank_float":
        chip = draw_chip((3, 3), blanks=[(1, 1)], dtype=np.float32, value=0.75)
        path = os.path.join(tempfile.mkdtemp(prefix="mgb_pinlist_"), "pinlist.csv")
        with open(path, "w") as f:
            f.write("Indices,MutantID\n")
            for i in range(3):
                for j in range(3):
                    f.write(f"\"({j + 1}, {i + 1})\",{'BLANK' if (i, j) == (1, 1) else f'm{i}{j}'}\n")
        data = xr.DataArray(data=chip, dims=("y", "x"))
        kw = dict(base, pinlist=path)
        return data, kw
    raise KeyError(case)


def draw_beads(shape, beads, value=1000, dtype=np.uint16):
    img = np.zeros(shape, dtype=dtype)
    for row, col, r in beads:
        pts = _disc(r)
        ok = (pts[:, 0] + row >= 0) & (pts[:, 0] + row < shape[0]) & (pts[:, 1] + col >= 0) & (pts[:, 1] + col < shape[1])
        img[pts[ok, 0] + row, pts[ok, 1] + col] = value
    return img


BEADS = [(60, 70, 9), (60, 200, 12), (150, 90, 7), (160, 300, 10), (250, 180, 11), (255, 199, 8), (300, 330, 9), (20, 360, 6)]


def bead_input(case):
    import xarray as xr

    base = dict(min_bead_diameter=10, max_bead_diameter=30, num_iter=1000, overlap=0)
    if case == "beads_single":
        frames = [draw_beads((360, 400), BEADS, 1000) + _noise((360, 400), 1), draw_beads((360, 400), BEADS[:5], 600) + _noise((360, 400), 2)]
        data = xr.DataArray(data=np.asarray(frames, dtype=np.uint16), dims=("channel", "y", "x"), coords={"channel": ["620", "435"]})
        return data, dict(base, search_channel="620")
    if case == "beads_flatfield_tiles":
        img = np.asarray([[draw_beads((360, 400), BEADS, 3000 + 500 * t) + 300 + _noise((360, 400), 5 + t) for t in range(2)]],
                         dtype=np.uint16)                                  # (channel=1, time=2, y, x)
        tiles = _split_tiles(img, 2, 2, 8)                                  # (1, 2, 2, 2, 188, 208)
        th, tw = tiles.shape[-2:]
        yy, xx = np.mgrid[0:th, 0:tw]
        flat = 0.8 + 0.4 * (yy / th) * (1 - xx / tw)
        dark = 100.0 + 10.0 * np.sin(xx / 17.0)
        data = xr.DataArray(data=tiles, dims=("channel", "time", "row", "col", "y", "x"))
        return data, dict(base, overlap=8, flatfield=flat, darkfield=dark)
    if case == "beads_none":
        data = xr.DataArray(data=np.zeros((2, 120, 130), dtype=np.uint16), dims=("channel", "y", "x"))
        return data, dict(base)
    raise KeyError(case)


def mrbles_input(tmpdir):
    """(DataArray, kwargs of mg.mrbles): 24 beads carrying three lanthanide codes (dy / eu volume
    ratio 0, 0.5, 1) seen through three channels, with the spectra and codes tables of
    identify_mrbles (identify.py:52-80) written as CSV files."""
    import xarray as xr

    channels = ["c435", "c546", "c620"]
    spectra = {"eu": [0.1, 0.2, 1.0], "dy": [0.9, 0.5, 0.1]}                  # rows: lanthanide, columns: channel
    ratios = {"code_a": 0.0, "code_b": 0.5, "code_c": 1.0}
    spectra_path, codes_path = os.path.join(tmpdir, "spectra.csv"), os.path.join(tmpdir, "codes.csv")
    with open(spectra_path, "w") as f:
        f.write("name," + ",".join(channels) + "\n")
        for ln in ("dy", "eu"):                                               # reference lanthanide deliberately not first
            f.write(ln + "," + ",".join(str(v) for v in spectra[ln]) + "\n")
    with open(codes_path, "w") as f:
        f.write("name,eu,dy\n")
        for name, r in ratios.items():
            f.write(f"{name},1.0,{r}\n")
    rng = np.random.default_rng(11)
    beads, values = [], []
    names = list(ratios)
    for i in range(4):
        for j in range(6):
            row, col, r = 45 + 70 * i + int(rng.integers(-5, 6)), 45 + 70 * j + int(rng.integers(-5, 6)), int(rng.integers(7, 12))
            beads.append((row, col, r))
            code = names[(i * 6 + j) % 3]
            vol_eu = 900.0 * (1 + 0.05 * rng.standard_normal())
            vol_dy = vol_eu * ratios[code] * (1 + 0.03 * rng.standard_normal())
            values.append([vol_eu * spectra["eu"][k] + vol_dy * spectra["dy"][k] for k in range(3)])
    frames = []
    for k in range(3):
        img = np.zeros((330, 470), dtype=np.float64)
        for (row, col, r), v in zip(beads, values):
            pts = _disc(r)
            img[pts[:, 0] + row, pts[:, 1] + col] = v[k]
        frames.append(img + 100 + _noise((330, 470), 20 + k, scale=10))
    data = xr.DataArray(data=np.asarray(frames).astype(np.uint16), dims=("channel", "y", "x"), coords={"channel": channels})
    kwargs = dict(spectra=spectra_path, codes=codes_path, min_bead_diameter=10, max_bead_diameter=30, num_iter=1000, overlap=0,
                  search_channel="c620", reference="eu")
    return data, kwargs


# ---------------------------------------------------------------------------------------------
# comparison
# ---------------------------------------------------------------------------------------------
def dataset_records(ds):
    """name -> (is_coord, dims, values) of every variable of a Dataset (ours or xarray's)."""
    coords = set(ds.coords)
    return {name: (name in coords, tuple(var.dims), np.asarray(var.values)) for name, var in ds.variables.items()}


def assert_same_dataset(got, want):
    assert type(got) is type(want), (type(got), type(want))
    g, w = dataset_records(got), dataset_records(want)
    assert set(g) == set(w), set(g) ^ set(w)
    for name in w:
        assert g[name][0] == w[name][0], f"{name}: coordinate on one side, data variable on the other"
        assert g[name][1] == w[name][1], f"{name}: dims {g[name][1]} != {w[name][1]}"
        a, b = g[name][2], w[name][2]
        assert a.dtype == b.dtype, f"{name}: dtype {a.dtype} != {b.dtype}"
        assert a.shape == b.shape, f"{name}: shape {a.shape} != {b.shape}"
        if a.dtype.kind == "f":
            np.testing.assert_array_equal(a, b, err_msg=name)       # NaN == NaN in assert_array_equal
        else:
            assert np.array_equal(a, b), f"{name}: values differ"
    assert set(got.attrs) == set(want.attrs), (set(got.attrs), set(want.attrs))
    for k in want.attrs:
        assert np.array_equal(np.asarray(got.attrs[k]), np.asarray(want.attrs[k])), f"attr {k}"


# ---------------------------------------------------------------------------------------------
# replay of the reference's pipeline states (tests/golden/dropin_*.npz)
# ---------------------------------------------------------------------------------------------
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_state(g, prefix):
    from magnify_b200.dataset import Dataset

    data, coords = {}, {}
    for entry in g[prefix + "__names"]:
        kind, name = str(entry).split(":", 1)
        dims = tuple(str(d) for d in g[f"{prefix}__{name}__dims"])
        (coords if kind == "coord" else data)[name] = (dims, g[f"{prefix}__{name}"])
    return Dataset(data, coords)


class Registry(dict):
    def register(self, name):
        return lambda f: self.__setitem__(name, f) or f

    def get(self, name):
        return self[name]


def run_pipe(components, assay):
    for _, component in components:          # pipeline.py:19-22
        assay = component(assay)
    return assay


def compare(got, want, names):
    for name in names:
        a, b = got[name], want[name]
        assert tuple(a.dims) == tuple(b.dims), (name, a.dims, b.dims)
        av, bv = np.asarray(a.values), np.asarray(b.values)
        assert av.dtype == bv.dtype and av.shape == bv.shape, (name, av.dtype, bv.dtype, av.shape, bv.shape)
        np.testing.assert_array_equal(av, bv, err_msg=name)
        assert (name in got.coords) == (name in want.coords), name


def replay_chip_case(case, on_device=True):
    """The chip components run on the `in__` state of tests/golden/dropin_<case>.npz must give
    its `out__` state, the reference-side summaries, and the `valid` flags of the three filters."""
    from magnify_b200 import components
    from magnify_b200.devarray import DeviceArray

    g = np.load(os.path.join(GOLDEN, f"dropin_{case}.npz"))
    kw = json.loads(str(g["kwargs_json"]))
    assay, want = load_state(g, "in"), load_state(g, "out")
    rows, cols = want["tag"].shape if want["tag"].ndim == 2 else (None, None)
    search = sorted(np.atleast_1d(kw["search_timestep"]).tolist())
    wx = np.asarray(want["x"].values)
    wy = np.asarray(want["y"].values)
    m = wx.shape[0]
    grid = (int(np.asarray(want["mark_row"].values).max()) + 1, int(np.asarray(want["mark_col"].values).max()) + 1)

    def centers(xp, t):
        k = search.index(t)
        return wx[:, t].reshape(grid), wy[:, t].reshape(grid), g["fg_radius"][k].reshape(grid)

    reg = Registry()
    components.install(registry=reg)
    finder_kw = {k: kw[k] for k in ("row_dist", "col_dist", "min_button_diameter", "max_button_diameter", "chamber_diameter",
                                    "top_chamber", "left_chamber", "low_edge_quantile", "high_edge_quantile", "num_iter",
                                    "min_roundness", "cluster_penalty", "roi_length", "progress_bar", "search_timestep",
                                    "search_channel", "interactive")}
    pipe = [("stitch", reg.get("stitch")(overlap=kw["overlap"])),
            ("find_buttons", reg.get("find_buttons")(**finder_kw, centers=centers))]
    got = run_pipe(pipe, assay)
    if on_device:
        assert isinstance(got["image"].data, DeviceArray) and isinstance(got["roi"].data, DeviceArray)   # nothing left the GPU yet
    assert got["roi"].shape[0] == m
    compare(got, want, ["image", "roi", "fg", "bg", "x", "y", "valid", "tag", "mark_row", "mark_col"])
    # and the summaries of the same pass equal the xarray expressions on the reference's dataset
    got = reg.get("quantify")()(got)
    if np.asarray(want["roi"].values).dtype == np.uint16:
        sel = want["roi"].where(want["fg"])
        np.testing.assert_array_equal(got["fg_median"].values, sel.median(dim=["roi_x", "roi_y"]).values)
        np.testing.assert_allclose(got["fg_mean"].values, sel.mean(dim=["roi_x", "roi_y"]).values, rtol=1e-6)
    # the consumers of the crops, in the order the golden generator ran the reference's own
    # (filter.py:11-94): medians and contour perimeters from the kernels, `valid` must follow exactly
    for name, fkw in (("filter_expression", {}), ("filter_nonround", {"min_roundness": 0.6}), ("filter_leaky", {})):
        got = reg.get(name)(**fkw)(got)
        np.testing.assert_array_equal(np.asarray(got["valid"].values), g[f"valid_after__{name}"], err_msg=name)


def replay_bead_case(case):
    """The bead components run on the `in__` state of tests/golden/dropin_<case>.npz must give its
    `out__` state."""
    from magnify_b200 import components

    g = np.load(os.path.join(GOLDEN, f"dropin_{case}.npz"))
    kw = json.loads(str(g["kwargs_json"]))
    assay, want = load_state(g, "in"), load_state(g, "out")
    beads = g["beads"]                       # the centres and radii the reference's (pinned) search returned
    reg = Registry()
    components.install(registry=reg)
    finder_kw = {k: kw[k] for k in ("min_bead_diameter", "max_bead_diameter", "low_edge_quantile", "high_edge_quantile",
                                    "num_iter", "min_roundness", "roi_length", "search_channel", "interactive")}
    pipe = []
    flat = g["kwarg__flatfield"] if "kwarg__flatfield" in g else kw["flatfield"]
    dark = g["kwarg__darkfield"] if "kwarg__darkfield" in g else kw["darkfield"]
    pipe.append(("flatfield_correct", reg.get("flatfield_correct")(flatfield=flat, darkfield=dark)))
    pipe.append(("stitch", reg.get("stitch")(overlap=kw["overlap"])))
    pipe.append(("find_beads", reg.get("find_beads")(**finder_kw, centers=beads)))
    got = run_pipe(pipe, assay)
    compare(got, want, ["image", "roi", "fg", "bg", "x", "y", "valid"])
