"""CPU-side checks: the C-ABI library builds, loads and exports every symbol the header
declares; host-side logic (argument errors, copy-forward map, disc table, fast-path fuzz)."""
import os
import re
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from magnify_b200.build import build_library
    from magnify_b200 import _lib

    build_library()
    return _lib.load()


def test_library_exports_header_symbols(lib):
    header = open(os.path.join(ROOT, "include", "magnify_b200.h")).read()
    declared = set(re.findall(r"\b(mgb_[a-z0-9_]+)\s*\(", header))
    assert len(declared) >= 18
    from magnify_b200 import _lib

    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.mgb_abi_version() == 12
    assert lib.mgb_error_string(-2).decode().startswith("pointer")


def test_sass_is_sm100a():
    so = os.path.join(ROOT, "magnify_b200", "libmagnify_b200.so")
    out = subprocess.run(["cuobjdump", "-lelf", so], capture_output=True, text=True)
    if out.returncode != 0:
        pytest.skip("cuobjdump unavailable")
    assert "sm_100a" in out.stdout
    # the staged gather really is TMA + mbarrier code, the masked sums really are dot-product
    # instructions (profiles/r02_sass_summary.md holds the per-kernel counts)
    sass = subprocess.run(["cuobjdump", "-sass", so], capture_output=True, text=True).stdout
    for mnemonic in ("UTMALDG", "SYNCS", "LDGSTS", "IDP.2A", "REDUX"):
        assert mnemonic in sass, mnemonic


def test_disc_halfwidths_host_entry_point(lib, golden):
    from magnify_b200 import ops

    d = golden("geometry")
    hw = d["disc_halfwidth"]
    table = ops.disc_halfwidth_table(hw.shape[0] - 1)
    for r in range(1, hw.shape[0]):
        np.testing.assert_array_equal(table[r, : r + 1], hw[r, : r + 1])
    import ctypes

    assert lib.mgb_disc_halfwidths(0, (ctypes.c_int32 * 1)()) == -1   # r = 0 raises in the reference


def test_argument_errors_before_any_launch(lib):
    """Validation happens on the host: these return a status without touching a GPU."""
    import ctypes

    p = ctypes.c_void_p(0)
    q16 = ctypes.c_void_p(4096)   # non-null and 16-byte aligned; never dereferenced, every call returns first
    assert lib.mgb_stitch(p, p, 0, 1, 1, 2, 2, 50, 50, -5, 2, None, p) == -1     # stitch.py:8-9
    assert lib.mgb_stitch(p, p, 0, 1, 1, 2, 2, 50, 50, 100, 2, None, p) == -1    # stitch.py:16-20
    assert lib.mgb_stitch(p, p, 0, 1, 1, 2, 2, 50, 50, 4, 3, None, p) == -1      # itemsize
    assert lib.mgb_stitch(p, p, 0, 0, 1, 2, 2, 50, 50, 4, 2, None, p) == 0       # empty: nothing to do
    assert lib.mgb_stitch(q16, q16, 10, 1, 1, 2, 2, 50, 56, 4, 2, None, p) == -1  # pitch < Cc * (W - overlap)

    ff = lib.mgb_flatfield_stitch_u16
    assert ff(p, p, 0, 1, 1, 2, 2, 50, 56, -5, 1, *[p] * 6) == -1                 # stitch.py:8-9
    assert ff(p, p, 0, 1, 1, 2, 2, 50, 56, 50, 1, *[p] * 6) == -1                 # stitch.py:16-20
    assert ff(p, p, 0, 0, 1, 2, 2, 50, 56, 4, 2, *[p] * 6) == -1                  # K neither 1 nor C
    assert ff(p, p, 0, 0, 1, 2, 2, 50, 56, 4, 1, *[p] * 6) == 0                   # empty: nothing to do
    assert ff(q16, q16, 0, 1, 1, 2, 2, 50, 56, 4, 1, *[q16] * 4, p, p) == -1      # null maxima table
    assert ff(q16, q16, 10, 1, 1, 2, 2, 50, 56, 4, 1, *[q16] * 6) == -1           # pitch < Cc * (W - overlap)
    assert ff(q16, q16, 0, 1, 1, 2, 2, 50, 52, 4, 1, *[q16] * 6) == -2            # W not whole 16-byte vectors

    # Size limits: mgb_stitch checks them before the empty-stack shortcut and the null pointers,
    # mgb_flatfield_stitch_u16 after them.
    tall = (2**31 - 1) // 8 + 1
    assert lib.mgb_stitch(p, p, 0, 0, 1, 2, 2, tall, 56, 4, 2, None, p) == -3
    assert ff(p, p, 0, 0, 1, 2, 2, tall, 56, 4, 1, *[p] * 6) == 0
    assert lib.mgb_stitch(p, p, 0, 1, 1, 2, 2, tall, 56, 4, 2, None, p) == -3
    assert ff(p, p, 0, 1, 1, 2, 2, tall, 56, 4, 1, *[p] * 6) == -1
    assert lib.mgb_stitch(q16, q16, 0, 1, 1, 2, 2, tall, 56, 4, 2, None, p) == -3
    assert ff(q16, q16, 0, 1, 1, 2, 2, tall, 56, 4, 1, *[q16] * 6) == -3
    assert lib.mgb_stitch(p, p, 0, 1, 1, 2**31, 0, 50, 56, 4, 2, None, p) == -3  # R > INT32_MAX, no tile columns
    assert ff(p, p, 0, 1, 1, 2**31, 0, 50, 56, 4, 1, *[p] * 6) == 0
    assert ff(p, p, 0, 70000, 0, 2, 2, 50, 56, 4, 70000, *[p] * 6) == 0           # K > 65535 tables
    assert ff(p, p, 0, 70000, 1, 2, 2, 50, 56, 4, 70000, *[p] * 6) == -1
    assert ff(q16, q16, 0, 70000, 1, 2, 2, 50, 56, 4, 70000, *[q16] * 6) == -3

    assert lib.mgb_bounding_boxes(p, p, 4, 72, 50, 50, p, p, p) == -1         # image smaller than box
    assert lib.mgb_roi_gather(p, 0, 1, 1, 100, 100, 2, p, p, 0, 72, p, p) == 0  # zero markers
    assert lib.mgb_chip_masks(p, p, 15, 30, 0, 72, p, p, p, p) == 0


def test_ops_refuse_cpu_tensors(lib):
    import torch
    from magnify_b200 import ops

    with pytest.raises(RuntimeError, match="CUDA"):
        ops.stitch(torch.zeros((1, 1, 1, 1, 8, 8), dtype=torch.uint16), 0)
    with pytest.raises(ValueError):
        ops.check_overlap(-1)
    with pytest.raises(ValueError):
        ops.check_overlap(10, 10, 12)


def test_copy_forward_sources_match_oracle():
    from magnify_b200.pipeline import copy_forward_sources
    from oracle.rois import chip_copy_forward

    for t, search in [(5, 0), (6, [2, 4]), (4, [3]), (7, [0, 3, 6]), (3, [1])]:
        np.testing.assert_array_equal(copy_forward_sources(t, search), chip_copy_forward(t, search))
    with pytest.raises(ValueError):
        copy_forward_sources(3, [5])


def test_flatfield_fast_path_fuzz_host(tmp_path):
    """The one-FMA fast path + guard band of ff_core.cuh, compiled for the host and fuzzed
    against the reference's exact operation order (20M pixels incl. degenerate coefficients)."""
    exe = tmp_path / "ff_fuzz"
    src = os.path.join(ROOT, "tests", "csrc", "ff_fuzz.cpp")
    subprocess.run(["g++", "-O2", "-o", str(exe), src], check=True)
    out = subprocess.run([str(exe), "20000000"], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout + out.stderr
    assert out.stdout.startswith("ok")


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    """No CPU fallback: without the built .so the binding raises instead of degrading."""
    from magnify_b200 import _lib

    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", str(tmp_path / "libmagnify_b200.so"))
    with pytest.raises(ImportError, match="no CPU fallback"):
        _lib.load()


def test_product_package_never_imports_the_oracle():
    """The oracle is test infrastructure: nothing under magnify_b200/ may import it."""
    import pathlib

    for path in pathlib.Path(ROOT, "magnify_b200").rglob("*.py"):
        text = path.read_text()
        assert "import oracle" not in text and "from oracle" not in text, path
