"""Host side of the TIFF staging row (SURVEY.md section 8f N2): the native page reader against
the struct-level oracle and OpenCV's libtiff, the path-pattern language against the reference's
own `extract_paths` run in place, and the assembly of the tile stack (reader.py:163-326).
File I/O only -- nothing here launches a kernel, so it runs without a GPU."""
import json
import os
import struct

import numpy as np
import pytest

from magnify_b200 import _lib, reader
from oracle import tiff as ot
from tiffgen import ome_xml, write_tiff


# ---- pages -----------------------------------------------------------------------------------
@pytest.mark.parametrize("big", [False, True])
@pytest.mark.parametrize("byteorder", ["<", ">"])
def test_native_pages_match_oracle(tmp_path, big, byteorder):
    rng = np.random.default_rng(0)
    for dtype in (np.uint8, np.uint16, np.int16, np.uint32, np.float32, np.float64):
        pages = [(rng.random((37, 53)) * 200).astype(dtype) for _ in range(4)]
        for rps, scatter in ((None, False), (5, False), (16, True), (1, True)):
            path = write_tiff(os.path.join(tmp_path, "a.tif"), pages, big=big, byteorder=byteorder, rows_per_strip=rps,
                              scatter=scatter, pad_strips=3 if scatter else 0, description="hello")
            with reader.TiffFile(path) as tif:
                assert tif.num_pages == 4
                info = tif.page_info(2)
                assert info.dtype == np.dtype(dtype) and info.shape == (37, 53)
                assert bool(info.bigtiff) == big and bool(info.big_endian) == (byteorder == ">")
                got = tif.read_pages([3, 0, 2], threads=3)
                for k, page in enumerate([3, 0, 2]):
                    np.testing.assert_array_equal(got[k], ot.read_page(path, page))
                    np.testing.assert_array_equal(got[k], pages[page])
                assert tif.description(0) == b"hello" and tif.description(1) == b""


def test_native_reads_libtiff_files_and_refuses_jpeg(tmp_path):
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(1)
    pages = [rng.integers(0, 65535, (64, 96), dtype=np.uint16) for _ in range(3)]
    multi = os.path.join(tmp_path, "m.tif")
    assert cv2.imwritemulti(multi, pages, [cv2.IMWRITE_TIFF_COMPRESSION, 1])
    with reader.TiffFile(multi) as tif:
        np.testing.assert_array_equal(tif.read_pages([0, 1, 2]), np.stack(pages))
    lzw = os.path.join(tmp_path, "lzw.tif")
    assert cv2.imwrite(lzw, pages[0])                                # libtiff default: LZW + differencing
    with reader.TiffFile(lzw) as tif:
        assert tif.page_info(0).compression == 5 and tif.page_info(0).status == 0
        np.testing.assert_array_equal(tif.asarray(0), pages[0])
    jpeg = os.path.join(tmp_path, "jpeg.tif")                        # JPEG-in-TIFF: not decoded here
    assert cv2.imwrite(jpeg, (pages[0] >> 8).astype(np.uint8), [cv2.IMWRITE_TIFF_COMPRESSION, 7])
    with reader.TiffFile(jpeg) as tif:
        assert tif.page_info(0).compression == 7 and tif.page_info(0).status == _lib.MGB_EUNSUPPORTED
        with pytest.raises(_lib.MagnifyB200Error) as err:
            tif.asarray(0)
        assert err.value.code == _lib.MGB_EUNSUPPORTED


def test_open_errors(tmp_path):
    bad = os.path.join(tmp_path, "bad.tif")
    open(bad, "wb").write(b"definitely not a tiff file")
    with pytest.raises(_lib.MagnifyB200Error) as err:
        reader.TiffFile(bad)
    assert err.value.code == _lib.MGB_EFORMAT
    with pytest.raises(_lib.MagnifyB200Error) as err:
        reader.TiffFile(os.path.join(tmp_path, "missing.tif"))
    assert err.value.code == _lib.MGB_EIO
    # truncated pixel data: the directory is fine, the strip runs past the end of the file
    page = np.arange(64 * 64, dtype=np.uint16).reshape(64, 64)
    cut = write_tiff(os.path.join(tmp_path, "cut.tif"), [page])
    raw = open(cut, "rb").read()
    ifd = struct.unpack("<I", raw[4:8])[0]
    # keep header + directory, drop half of the pixel bytes by rewriting them past EOF
    with open(cut, "wb") as f:
        f.write(raw[:8] + raw[8 + 4096:])
    with pytest.raises(_lib.MagnifyB200Error):
        with reader.TiffFile(cut) as tif:
            tif.asarray(0)
    assert ifd > 8
    with pytest.raises(ValueError):
        ok = write_tiff(os.path.join(tmp_path, "ok.tif"), [page])
        with reader.TiffFile(ok) as tif:
            tif.read_pages([0], out=np.empty((1, 64, 64), np.float32))


def test_read_files_checks_geometry(tmp_path):
    rng = np.random.default_rng(2)
    pages = [rng.integers(0, 65535, (32, 48), dtype=np.uint16) for _ in range(5)]
    paths = [write_tiff(os.path.join(tmp_path, f"t{i}.tif"), [p], big=bool(i % 2), byteorder="<>"[i % 2],
                        rows_per_strip=[None, 3, 32, 7, 1][i]) for i, p in enumerate(pages)]
    out = np.empty((5, 32, 48), np.uint16)
    reader.read_files(paths, out, threads=3)
    np.testing.assert_array_equal(out, np.stack(pages))
    odd = write_tiff(os.path.join(tmp_path, "odd.tif"), [pages[0][:, :40]])
    with pytest.raises(_lib.MagnifyB200Error) as err:
        reader.read_files(paths[:2] + [odd], np.empty((3, 32, 48), np.uint16))
    assert err.value.code == _lib.MGB_EFORMAT


# ---- path patterns ---------------------------------------------------------------------------
KEYS = dict(assay="str", channel="str", time="time", row="int", col="int")


def make_tree(root):
    for assay in ("xpA", "xpB"):
        for ch in ("egfp", "Cy5"):
            os.makedirs(os.path.join(root, assay, ch), exist_ok=True)
            for t in ("20240101-120000", "20240101-130000"):
                for r in range(2):
                    for c in range(3):
                        open(os.path.join(root, assay, ch, f"img_{t}_{r}_{c}_conc{1.5 * r}.tif"), "w").close()
    os.makedirs(os.path.join(root, "flat"))
    for i in range(3):
        open(os.path.join(root, "flat", f"tile{i}.TIF"), "w").close()


def patterns(root):
    return [f"{root}/(assay)/(channel)/img_(time)_(row)_(col)_conc(conc_row|float).tif",
            f"{root}/(assay)/(channel)/img_(time|%Y%m%d-%H%M%S)_(row)_(col)_*.tif",
            f"{root}/xpA/(channel)/img_20240101-120000_(row)_(col)_*.tif",
            f"{root}/xpB/egfp/img_(time | %Y%m%d-%H%M%S)_1_(col)_conc(amount_col|float).tif",
            f"{root}/flat/tile(col).TIF",
            f"{root}/flat/*.TIF",
            f"{root}/**/img_(time)_0_(col)_conc0.0.tif",
            f"{root}/nothing/(row).tif"]


def outcome(fn, pattern):
    try:
        paths, meta = fn(pattern, **KEYS)
        return paths, {k: dict(v) for k, v in meta.items()}
    except Exception as e:   # noqa: BLE001 -- the exception type is the outcome
        return type(e).__name__


def test_extract_paths_contract(tmp_path):
    make_tree(str(tmp_path))
    import datetime

    paths, meta = reader.extract_paths(patterns(str(tmp_path))[0], **KEYS)
    assert len(paths) == 48
    key = ("xpA", "Cy5", datetime.datetime(2024, 1, 1, 13, 0), 1, 2)
    assert paths[key].endswith("xpA/Cy5/img_20240101-130000_1_2_conc1.5.tif")
    assert dict(meta["conc", "row"]) == {0: 0.0, 1: 1.5}
    paths, _ = reader.extract_paths(patterns(str(tmp_path))[2], **KEYS)
    assert len(paths) == 12 and all(k[0] is None and k[2] is None for k in paths)
    with pytest.raises(ValueError):
        reader.extract_paths(patterns(str(tmp_path))[5], **KEYS)


def canonical_outcome(fn, root):
    """repr of each pattern's outcome with its mappings in sorted order and the tree's root
    written as <root>."""
    def canonical(result):
        if isinstance(result, str):
            return result
        paths, meta = result
        return (sorted(paths.items(), key=repr), sorted(((k, sorted(v.items(), key=repr)) for k, v in meta.items()), key=repr))

    return [repr(canonical(outcome(fn, pattern))).replace(root, "<root>") for pattern in patterns(root)]


def record(tmpdir):
    """This package's side of the comparison with the reference's extract_paths (written to
    tests/golden/reference_record.npz by tests/golden/make_reference_record.py)."""
    make_tree(tmpdir)
    return {"extract_paths": np.array(canonical_outcome(reader.extract_paths, tmpdir))}


def test_extract_paths_against_reference_source_when_present(tmp_path, golden):
    """What the reference's extract_paths returned (tests/golden/reference_record.npz), and the
    reference itself when it is present."""
    from oracle._refload import load_reference_reader

    want = [str(v) for v in golden("reference_record")["extract_paths"]]
    make_tree(str(tmp_path))
    assert canonical_outcome(reader.extract_paths, str(tmp_path)) == want
    ref = load_reference_reader()
    if ref is not None:
        assert canonical_outcome(ref.extract_paths, str(tmp_path)) == want


# ---- tile stack assembly ---------------------------------------------------------------------
def test_read_tiffs_file_per_index(tmp_path):
    rng = np.random.default_rng(3)
    c, t, r, cc, h, w = 2, 3, 2, 2, 24, 32
    tiles = rng.integers(0, 65535, (c, t, r, cc, h, w), dtype=np.uint16)
    chs, stamps = ["cy5", "egfp"], ["20240101-120000", "20240101-120100", "20240101-120200"]
    for idx in np.ndindex(c, t, r, cc):
        write_tiff(os.path.join(tmp_path, f"xp_{chs[idx[0]]}_{stamps[idx[1]]}_{idx[2]}_{idx[3]}.tif"), [tiles[idx]],
                   rows_per_strip=7)
    (xp,) = list(reader.Reader(threads=3)(os.path.join(tmp_path, "xp_(channel)_(time)_(row)_(col).tif")))
    assert xp["tile"].dims == reader.TILE_ORDER and xp["tile"].shape == tiles.shape
    np.testing.assert_array_equal(np.asarray(xp["tile"]), tiles)
    np.testing.assert_array_equal(xp["tile"].data.read((1, 2)), tiles[1, 2])
    assert list(xp.coords["channel"].values) == chs
    assert np.diff(xp.coords["time"].values).tolist() == [60, 60]
    blocks = dict(xp["tile"].data.blocks())
    dst = np.empty((r, cc, h, w), np.uint16)
    blocks[(0, 1)](dst)
    np.testing.assert_array_equal(dst, tiles[0, 1])
    # rows / cols only in the path: standardize_format adds channel and time (preprocess.py:35-40)
    (xp2,) = list(reader.Reader()(os.path.join(tmp_path, "xp_cy5_20240101-120000_(row)_(col).tif")))
    assert xp2["tile"].dims == ("tile_row", "tile_col", "tile_y", "tile_x")
    std = reader.standardize_format(xp2)
    assert std["tile"].dims == reader.TILE_ORDER and std["tile"].shape == (1, 1, r, cc, h, w)
    assert std.attrs["__original_tile_dims__"] == ["tile_row", "tile_col", "tile_y", "tile_x"]
    np.testing.assert_array_equal(np.asarray(std["tile"])[0, 0], tiles[0, 0])
    with pytest.raises(FileNotFoundError):
        list(reader.Reader()(os.path.join(tmp_path, "nothing_(row).tif")))


def test_read_tiffs_ome_series_with_micromanager_summary(tmp_path):
    rng = np.random.default_rng(4)
    c, t, h, w = 2, 3, 24, 32
    planes = rng.integers(0, 65535, (t, c, h, w), dtype=np.uint16)
    summary = json.dumps({"StartTime": "2024-01-01 12:00:00.000 -0800", "ChNames": ["a", "b"]}).encode()
    header = struct.pack("<IIIIII", 54773648, 0, 483765892, 0, 99384722, 0) + struct.pack("<II", 2355492, len(summary)) \
        + summary
    xml = ome_xml(w, h, c, t, order="XYCZT", delta_t_ms=[1000.0 * i for i in range(c * t)])
    for row in range(2):
        pages = [planes[ti, ci] if row == 0 else planes[ti, ci][::-1] for ti in range(t) for ci in range(c)]
        write_tiff(os.path.join(tmp_path, f"ome_{row}.ome.tif"), pages, description=xml, header_extra=header)
    (xp,) = list(reader.Reader()(os.path.join(tmp_path, "ome_(row).ome.tif")))
    assert xp["tile"].dims == ("channel", "time", "tile_row", "tile_y", "tile_x")
    arr = np.asarray(xp["tile"])
    np.testing.assert_array_equal(arr[:, :, 0], planes.transpose(1, 0, 2, 3))
    np.testing.assert_array_equal(arr[:, :, 1], planes.transpose(1, 0, 2, 3)[:, :, ::-1])
    assert list(xp.coords["channel"].values) == ["a", "b"]
    assert np.diff(xp.coords["time"].values).tolist() == [2, 2]      # DeltaT of every c-th plane
    std = reader.standardize_format(xp)
    np.testing.assert_array_equal(std["tile"].data.read((1, 2)), arr[1, 2][:, None])
    # a multi-page file without OME-XML has the series axis "I": unmappable, like reader.py:208
    write_tiff(os.path.join(tmp_path, "plain_0.tif"), [planes[0, 0], planes[0, 1]])
    with pytest.raises(KeyError):
        list(reader.Reader()(os.path.join(tmp_path, "plain_(row).tif")))


def test_corrupted_files_never_crash_the_reader(tmp_path):
    """Byte flips and truncations in the header / directory of valid files: the native parser
    either reads the file or reports an error code -- no crash, no hang, no huge allocation."""
    rng = np.random.default_rng(7)
    page = rng.integers(0, 65535, (40, 48), dtype=np.uint16)
    outcomes = {"ok": 0, "error": 0}
    for big in (False, True):
        for byteorder in "<>":
            good = write_tiff(os.path.join(tmp_path, "g.tif"), [page, page[::-1]], big=big, byteorder=byteorder,
                              rows_per_strip=7, description="d" * 40)
            raw = bytearray(open(good, "rb").read())
            ifd_region = list(range(0, 16)) + list(range(len(raw) - 700, len(raw)))
            for trial in range(150):
                bad = bytearray(raw)
                if trial % 5 == 0:
                    bad = bad[: int(rng.integers(1, len(bad)))]
                else:
                    for _ in range(int(rng.integers(1, 6))):
                        pos = int(rng.choice(ifd_region))
                        if pos < len(bad):
                            bad[pos] = int(rng.integers(0, 256))
                path = os.path.join(tmp_path, "b.tif")
                open(path, "wb").write(bytes(bad))
                try:
                    with reader.TiffFile(path) as tif:
                        for k in range(min(tif.num_pages, 3)):
                            info = tif.page_info(k)
                            if info.status == 0 and 0 < info.nbytes < (1 << 24):
                                tif.read_pages([k], out=np.empty((1,) + info.shape, info.dtype), threads=1)
                            tif.description(k)
                    outcomes["ok"] += 1
                except _lib.MagnifyB200Error:
                    outcomes["error"] += 1
    assert outcomes["ok"] > 0 and outcomes["error"] > 0


# ---- compressed / differenced / tiled pages ---------------------------------------------------
def test_libtiff_compressed_files_decode(tmp_path):
    """Files written by libtiff through cv2.imwrite with LZW (its default, with horizontal
    differencing), Deflate and PackBits: the native decoders reproduce the pixels."""
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(5)
    smooth = (np.add.outer(np.arange(300), np.arange(257)) * 37 % 60000).astype(np.uint16)
    images = [smooth, rng.integers(0, 65535, (123, 131), dtype=np.uint16), (smooth >> 8).astype(np.uint8),
              np.zeros((64, 64), np.uint16), rng.integers(0, 255, (50, 70), dtype=np.uint8)]
    for k, img in enumerate(images):
        for comp in (5, 8, 32946, 32773, 1):
            path = os.path.join(tmp_path, f"c{k}_{comp}.tif")
            assert cv2.imwrite(path, img, [cv2.IMWRITE_TIFF_COMPRESSION, comp])
            with reader.TiffFile(path) as tif:
                info = tif.page_info(0)
                assert info.status == 0 and info.compression == comp
                np.testing.assert_array_equal(tif.asarray(0), img, err_msg=f"image {k} compression {comp}")
            np.testing.assert_array_equal(cv2.imread(path, cv2.IMREAD_UNCHANGED), img)
    multi = os.path.join(tmp_path, "multi_lzw.tif")
    assert cv2.imwritemulti(multi, images[:2] and [smooth, smooth[::-1].copy()])
    with reader.TiffFile(multi) as tif:
        got = tif.read_pages([1, 0], threads=2)
        np.testing.assert_array_equal(got[0], smooth[::-1])
        np.testing.assert_array_equal(got[1], smooth)


@pytest.mark.parametrize("big", [False, True])
@pytest.mark.parametrize("byteorder", ["<", ">"])
def test_tiled_deflate_and_predictor_pages(tmp_path, big, byteorder):
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(6)
    for dtype in (np.uint8, np.uint16, np.uint32, np.float32):
        page = (rng.random((70, 90)) * 200).astype(dtype)
        for kw in (dict(tile=(16, 32)), dict(tile=(64, 64), deflate=True), dict(deflate=True, rows_per_strip=9),
                   dict(deflate=True, predictor=True, rows_per_strip=16), dict(tile=(32, 16), deflate=True, predictor=True)):
            if kw.get("predictor") and np.dtype(dtype).kind == "f":
                continue
            path = write_tiff(os.path.join(tmp_path, "t.tif"), [page, page.T.copy()], big=big, byteorder=byteorder, **kw)
            with reader.TiffFile(path) as tif:
                np.testing.assert_array_equal(tif.asarray(0), page, err_msg=str(kw))
                np.testing.assert_array_equal(tif.asarray(1), page.T, err_msg=str(kw))
            if dtype != np.uint32:                                  # libtiff through OpenCV agrees with the writer
                ok, decoded = cv2.imreadmulti(path, flags=cv2.IMREAD_UNCHANGED)
                assert ok and np.array_equal(decoded[0], page)


def test_corrupt_compressed_data_is_an_error(tmp_path):
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(8)
    img = rng.integers(0, 65535, (64, 64), dtype=np.uint16)
    for comp in (5, 8, 32773):
        path = os.path.join(tmp_path, f"x{comp}.tif")
        assert cv2.imwrite(path, img, [cv2.IMWRITE_TIFF_COMPRESSION, comp])
        raw = bytearray(open(path, "rb").read())
        for trial in range(40):
            bad = bytearray(raw)
            for _ in range(4):
                bad[int(rng.integers(8, len(bad) - 300))] = int(rng.integers(0, 256))
            open(path, "wb").write(bytes(bad))
            try:
                with reader.TiffFile(path) as tif:
                    tif.asarray(0)                                   # wrong pixels are acceptable, a crash is not
            except _lib.MagnifyB200Error:
                pass


def test_write_tiff_round_trip(tmp_path):
    """reader.write_tiff -> the native reader, the struct-level oracle and libtiff all read the same pages."""
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(9)
    for dtype in (np.uint8, np.uint16, np.int16, np.float32, np.float64):
        pages = (rng.random((3, 45, 67)) * 200).astype(dtype)
        for big, desc in ((False, None), (True, "stitched image, channel egfp"), (None, "x")):
            path = reader.write_tiff(os.path.join(tmp_path, "w.tif"), pages, description=desc, bigtiff=big, threads=3)
            with reader.TiffFile(path) as tif:
                assert tif.num_pages == 3 and bool(tif.page_info(0).bigtiff) == bool(big)
                np.testing.assert_array_equal(tif.read_pages([0, 1, 2]), pages)
                assert tif.description(0) == (desc.encode() if desc else b"")
            for k in range(3):
                np.testing.assert_array_equal(ot.read_page(path, k), pages[k])
            if dtype != np.float64 and dtype != np.int16:
                ok, decoded = cv2.imreadmulti(path, flags=cv2.IMREAD_UNCHANGED)
                assert ok and len(decoded) == 3 and np.array_equal(np.stack(decoded), pages)
    single = reader.write_tiff(os.path.join(tmp_path, "s.tif"), pages[0])
    with reader.TiffFile(single) as tif:
        assert tif.num_pages == 1
    with pytest.raises(ValueError):
        reader.write_tiff(os.path.join(tmp_path, "bad.tif"), np.zeros((2, 2, 2, 2), np.uint8))
    with pytest.raises(_lib.MagnifyB200Error):
        reader.write_tiff(os.path.join(tmp_path, "no_such_dir", "x.tif"), pages)


def test_written_tiles_read_back_through_the_pattern_reader(tmp_path):
    """reader.write_tiff + reader.Reader: a tile stack saved page by page comes back as the same
    lazy (channel, time, tile_row, tile_col, tile_y, tile_x) array."""
    rng = np.random.default_rng(10)
    tiles = rng.integers(0, 65535, (2, 2, 2, 3, 20, 28), dtype=np.uint16)
    for idx in np.ndindex(2, 2, 2, 3):
        reader.write_tiff(os.path.join(tmp_path, f"w_c{idx[0]}_2024010{idx[1] + 1}-000000_{idx[2]}_{idx[3]}.tif"), tiles[idx])
    (xp,) = list(reader.Reader(threads=2)(os.path.join(tmp_path, "w_(channel)_(time)_(row)_(col).tif")))
    np.testing.assert_array_equal(np.asarray(xp["tile"]), tiles)
