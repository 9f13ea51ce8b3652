"""Every launch configuration of the stitch and flat-field + stitch kernels against the float64 oracle.

`mgb_stitch` (MODE 0, a copy of any 2/4/8-byte element as 16-bit units) and
`mgb_flatfield_stitch_u16` (MODE 1) launch `stitch_u16_kernel` with a host-side plan: the tile
column period P of the output phase (clamped to the tile columns), the input shift S of each
phase slice, the number of 2048-unit x-blocks, and the split of the image loop over CTAs
(`ct_splits`).  Inside the kernel, whole warps right of the kept row return early, lane 31 of a
warp streams one extra input chunk for its shifted vector, the first vector of a row may start
left of the tile, and the per-CTA loop may be shorter than the prefetch ring.  When the
alignment conditions fail, `mgb_stitch` takes the element-wise kernel and the flat-field entry
answers MGB_EALIGN, after which `ops.flatfield_stitch` applies the exact generic kernel and
stitches.

`stitch_plan` restates that host logic.  Every case of the matrix names the plan features it
is meant to reach and asserts them, so a case that drifts away from its purpose fails.  Each
case calls the C entry points directly (which path ran is asserted), writes into an output
buffer whose row padding and surrounding guard bytes hold a sentinel, and compares the raw
buffer bit for bit with `oracle.stitch.stitch` / `oracle.flatfield.flatfield_correct`.  Each
case runs under the three stitch variants (prefetch-ring depth x CTAs per SM).  The maxima pass
(`flatfield_maxima`, `flatfield_maxima_accumulate`) is compared with
`oracle.flatfield.flatfield_maxima` bit for bit.

`test_matrix_covers_every_launch_feature` needs no GPU: it checks, from the case list and the
plan alone, that the matrix reaches every (P, S) in both modes and every other feature above.
"""
import ctypes
import math
from collections import namedtuple

import numpy as np
import pytest
import torch

from oracle import flatfield as o_ff
from oracle import stitch as o_st

gpu = pytest.mark.gpu

STAGES = {0: 6, 1: 11, 2: 8}     # mgb_set_stitch_variant -> prefetch-ring stages
TARGET_ITERS = {0: 32, 1: 160}   # per-CTA tile loop the launcher aims for, per MODE
B200_SMS = 148
SENTINEL = 0xA5

# ------------------------------------------------------------------------------ launch plan
Plan = namedtuple("Plan", "fast u P P_unclamped xblocks launches ct_splits splits_wanted n_iters "
                          "early_return lane31 a0_neg spill uneven")


def stitch_plan(shape, overlap, itemsize, K, sm_count, target_iters, pitch=None, aligned=True):
    """The host logic of mgb_stitch / mgb_flatfield_stitch_u16 and run_stitch_fast restated.

    shape (C,T,R,Cc,H,W) in elements; pitch: image row pitch in elements (None: dense);
    aligned: tiles and image both start on 16-byte boundaries.  For the flat-field entry
    (uint16 only) `fast` False means MGB_EALIGN.  launches: set of (q, phase, S) in 16-bit
    units; n_iters: the set of per-CTA tile-loop lengths of CTAs that run the loop."""
    C, T, R, Cc, H, W = shape
    h, w = H - overlap, W - overlap
    clip = overlap // 2
    pitch = Cc * w if pitch is None else pitch
    fast = itemsize >= 2 and (W * itemsize) % 16 == 0 and (pitch * itemsize) % 16 == 0 and aligned
    if not fast:
        return Plan(False, None, None, None, None, frozenset(), None, None, frozenset(), False, False, False,
                    False, False)
    u = itemsize // 2
    wu, clip_u = w * u, clip * u
    wm = wu & 7
    p_unclamped = 8 // math.gcd(wm, 8) if wm else 1
    P = min(p_unclamped, Cc)
    xblocks = -(-(-(-(wu + 7) // 8)) // 256)
    launches = frozenset((q, (q * wu) & 7, (clip_u - ((q * wu) & 7)) % 8) for q in range(P))

    n_ct = C * T if K == 1 else T
    iters_per_ct = R * (-(-Cc // P))
    base_ctas = h * xblocks * K * P
    splits = -(-(n_ct * iters_per_ct) // target_iters)
    while base_ctas * splits < sm_count * 16 and (n_ct // (splits + 1)) * iters_per_ct >= 16:
        splits += 1
    wanted = splits
    splits = max(1, min(splits, n_ct, 32768))
    per_split = {n_ct * (s + 1) // splits - n_ct * s // splits for s in range(splits)}
    n_iters = frozenset(n * R * ((Cc - q + P - 1) // P) for n in per_split for q in range(P))

    early = lane31 = a0_neg = spill = False
    for _, phase, S in launches:
        a0_neg |= clip_u - phase < 0                      # thread 0: xin0 = clip - phase
        for xb in range(xblocks):
            spill |= xb > 0 and 8 * xb * 256 - phase < wu
            for warp in range(8):
                j0 = xb * 256 + warp * 32
                if 8 * j0 - phase >= wu:                      # the whole warp returns
                    early = True
                    continue
                xk0 = 8 * (j0 + 31) - phase                   # lane 31
                # active, and its extra chunk (the last S units of its vector) reaches a stored pixel
                lane31 |= S != 0 and xk0 < wu and xk0 + 8 - S < wu
    return Plan(True, u, P, p_unclamped, xblocks, launches, splits, wanted, n_iters, early, lane31, a0_neg,
                spill, len(per_split) > 1)


def plan_features(plan, pitch, wim):
    """The named features of a plan (what a case can claim to reach)."""
    if not plan.fast:
        return {"generic"}
    f = {f"P{plan.P}", f"u{plan.u}", f"xb{min(plan.xblocks, 2)}"}
    if plan.P < plan.P_unclamped:
        f.add("Pclamp")
    if {s for _, _, s in plan.launches} == set(range(8)):
        f.add("allS")
    for flag in ("early_return", "lane31", "a0_neg", "spill", "uneven"):
        if getattr(plan, flag):
            f.add(flag)
    if plan.ct_splits > 1:
        f.add("split")
    if plan.splits_wanted > 32768:
        f.add("clamp32768")
    if len(plan.n_iters) == 1:
        f.add(f"iters{next(iter(plan.n_iters))}")
    if pitch > wim:
        f.add("padded")
    return f


# ---------------------------------------------------------------------------- case matrix
Case = namedtuple("Case", "mode dtype shape overlap layout iters kc toff features")

# uint16 geometries run in both modes: (shape, overlap, output layout, MGB_STITCH_ITERS, features)
U16_GEOMETRIES = [
    # P = 8 (odd kept width): every S in one launch, lane 31 active (kept row > 248), a0 < 0
    ((1, 2, 1, 8, 12, 272), 7, "pitch64", None, {"P8", "allS", "lane31", "a0_neg", "early_return", "padded"}),
    ((2, 1, 2, 9, 10, 272), 7, "alloc", None, {"P8", "allS", "lane31", "padded"}),
    ((1, 1, 1, 8, 14, 272), 9, "off16", None, {"P8", "allS", "lane31"}),
    # P = 4 from w % 8 in {2, 6} (odd S), and P = 8 clamped to Cc = 4 (S 0..3, 4..7)
    ((1, 2, 1, 4, 12, 64), 6, "dense", None, {"P4"}),
    ((1, 1, 2, 6, 12, 64), 2, "alloc", None, {"P4", "padded"}),
    ((1, 1, 1, 4, 12, 272), 7, "alloc", None, {"P4", "Pclamp", "lane31", "padded"}),
    ((1, 1, 1, 4, 20, 272), 15, "alloc", None, {"P4", "Pclamp", "lane31"}),
    # P = 2 from w % 8 == 4, and P = 8 clamped to Cc = 2 at several clips
    ((1, 2, 1, 2, 12, 64), 4, "dense", None, {"P2"}),
    ((1, 1, 2, 2, 12, 272), 1, "alloc", None, {"P2", "Pclamp"}),
    ((1, 1, 1, 2, 12, 272), 9, "alloc", None, {"P2", "Pclamp"}),
    ((1, 1, 1, 2, 16, 272), 13, "alloc", None, {"P2", "Pclamp"}),
    ((1, 1, 1, 2, 18, 272), 15, "off16", None, {"P2", "Pclamp"}),
    # P = 1 from w % 8 == 0
    ((1, 2, 2, 3, 12, 64), 0, "dense", None, {"P1"}),
    ((1, 1, 1, 3, 16, 64), 8, "pitch64", None, {"P1", "padded"}),
    # tiny kept widths 7..1 (W = 8), nine tile columns: P = 8 for odd widths, Cc < P for P = 1, 2, 4
    *[((1, 2, 2, 9, 8, 8), ov, "alloc", None, {"xb1", "early_return", "a0_neg", "padded"}) for ov in range(1, 8)],
    # x-block boundary: w = 2041 fills one block at phase 7; w = 2043 spills phases 6, 7 into a
    # second block; w = 2042 launches a second block whose warps all return
    ((1, 1, 1, 8, 10, 2048), 7, "alloc", None, {"P8", "allS", "xb1"}),
    ((1, 1, 1, 8, 10, 2048), 5, "alloc", None, {"P8", "allS", "xb2", "spill"}),
    ((1, 1, 1, 4, 10, 2048), 6, "pitch64", None, {"P4", "xb2", "early_return"}),
    # per-CTA loop of exactly 1, 5..12 tiles (stages - 1, stages, stages + 1 of every variant);
    # Cc = 1 clamps P to 1 and overlaps 1..15 give every clip, so every S with P = 1
    *[((1, 2, n, 1, 24, 24), 2 * (i % 8) + 1, "alloc", 1, {"P1", f"iters{n}"})
      for i, n in enumerate((1, 5, 6, 7, 8, 9, 10, 11, 12))],
    # ct_splits: uneven split of 7 images over 3 CTAs; the 16 x SMs loop; the 32768 clamp
    ((1, 7, 2, 3, 12, 64), 6, "alloc", 5, {"split", "uneven"}),
    ((2, 20, 4, 2, 12, 64), 4, "dense", None, {"split"}),
    ((1, 40000, 1, 1, 2, 8), 1, "alloc", 1, {"split", "uneven", "clamp32768"}),
]


def _cases():
    cases = []
    for shape, ov, layout, iters, feat in U16_GEOMETRIES:
        for mode in (0, 1):
            cases.append(Case(mode, "uint16", shape, ov, layout, iters, False, 0, frozenset(feat | {"u1"})))
    cases += [
        # element sizes of the plain stitch: 4- and 8-byte elements as 2 and 4 units
        Case(0, "float32", (1, 2, 1, 5, 10, 64), 3, "alloc", None, False, 0, frozenset({"u2", "P4"})),
        Case(0, "float32", (1, 1, 1, 4, 9, 1024), 1, "alloc", None, False, 0, frozenset({"u2", "P4", "xb2", "spill"})),
        Case(0, "float64", (1, 1, 2, 3, 9, 34), 3, "alloc", None, False, 0, frozenset({"u4", "P2"})),
        Case(0, "float64", (2, 1, 1, 2, 9, 40), 0, "pitch64", None, False, 0, frozenset({"u4", "P1", "padded"})),
        # rows of W * itemsize not a multiple of 16 bytes, 1-byte elements, misaligned pointers:
        # the element-wise kernel
        Case(0, "uint16", (1, 2, 1, 3, 10, 20), 3, "alloc", None, False, 0, frozenset({"generic"})),
        Case(0, "float32", (1, 2, 1, 3, 10, 30), 3, "alloc", None, False, 0, frozenset({"generic"})),
        Case(0, "float64", (1, 1, 1, 3, 9, 33), 2, "alloc", None, False, 0, frozenset({"generic"})),
        Case(0, "uint8", (1, 2, 2, 3, 12, 32), 5, "alloc", None, False, 0, frozenset({"generic"})),
        Case(0, "uint16", (1, 2, 1, 8, 12, 272), 7, "alloc", None, False, 1, frozenset({"generic"})),
        Case(0, "float32", (1, 1, 1, 5, 10, 64), 3, "alloc", None, False, 2, frozenset({"generic"})),
        Case(0, "uint16", (1, 2, 1, 8, 12, 272), 7, "off1el", None, False, 0, frozenset({"generic"})),
        Case(0, "float64", (1, 1, 2, 3, 9, 34), 3, "off1el", None, False, 0, frozenset({"generic"})),
        Case(0, "uint16", (1, 2, 2, 9, 8, 8), 3, "dense", None, False, 0, frozenset({"generic"})),
        # flat-field: MGB_EALIGN -> exact generic kernel + stitch
        Case(1, "uint16", (1, 2, 1, 8, 12, 272), 7, "alloc", None, False, 1, frozenset({"generic"})),
        Case(1, "uint16", (1, 2, 1, 8, 12, 272), 7, "off1el", None, False, 0, frozenset({"generic"})),
        Case(1, "uint16", (1, 2, 1, 3, 10, 20), 3, "alloc", None, False, 0, frozenset({"generic"})),
        Case(1, "uint16", (1, 2, 2, 9, 8, 8), 3, "dense", None, False, 0, frozenset({"generic"})),
        # per-channel tables (K = C) with the image loop split over CTAs
        Case(1, "uint16", (3, 5, 1, 2, 12, 64), 6, "alloc", 3, True, 0, frozenset({"split", "uneven"})),
        Case(1, "uint16", (3, 6, 2, 9, 10, 272), 7, "alloc", 4, True, 0, frozenset({"P8", "allS", "split"})),
        Case(1, "uint16", (4, 5, 2, 2, 12, 64), 4, "dense", None, True, 0, frozenset({"P2"})),
    ]
    return cases


CASES = _cases()


def _case_id(case):
    c, t, r, cc, h, w = case.shape
    s = f"m{case.mode}-{case.dtype}-{c}x{t}x{r}x{cc}x{h}x{w}-ov{case.overlap}-{case.layout}"
    if case.iters:
        s += f"-it{case.iters}"
    if case.kc:
        s += "-KC"
    if case.toff:
        s += f"-toff{case.toff}"
    return s


def _layout(case_or_layout, wim, itemsize):
    """(pitch, byte offset of the image in its buffer) of an output layout."""
    layout = getattr(case_or_layout, "layout", case_or_layout)
    quantum = max(1, 16 // itemsize)
    padded = -(-wim // quantum) * quantum
    pitch = {"dense": wim, "alloc": padded, "pitch64": wim + 64, "off16": padded, "off1el": padded}[layout]
    front = {"off16": 16, "off1el": 256 + itemsize}.get(layout, 256)
    return pitch, front


def case_plan(case, sm_count):
    itemsize = np.dtype(case.dtype).itemsize
    C, T, R, Cc, H, W = case.shape
    wim = Cc * (W - case.overlap)
    pitch, front = _layout(case, wim, itemsize)
    aligned = front % 16 == 0 and (case.toff * itemsize) % 16 == 0
    target = case.iters or TARGET_ITERS[case.mode]
    plan = stitch_plan(case.shape, case.overlap, itemsize, C if case.kc else 1, sm_count, target, pitch, aligned)
    return plan, pitch, wim


def _check_case_features(case, sm_count):
    plan, pitch, wim = case_plan(case, sm_count)
    got = plan_features(plan, pitch, wim)
    missing = set(case.features) - got
    assert not missing, f"{_case_id(case)} no longer reaches {sorted(missing)} (plan features {sorted(got)})"
    return plan, got


def test_matrix_covers_every_launch_feature():
    """No GPU: from the case list and stitch_plan on a 148-SM B200, the matrix reaches every
    (P, S) in both modes, 16-bit units per element 1, 2 and 4, one and two x-blocks with an
    active vector in the second, early warp returns, an active lane 31 with S != 0, a0 < 0,
    per-CTA loops of 1, stages - 1, stages and stages + 1 for every variant, uneven ct_splits,
    per-channel tables with a split loop, padded pitches, and the generic paths of both modes."""
    seen = {0: set(), 1: set()}
    pairs = {0: set(), 1: set()}
    iters = set()
    kc_split = False
    for case in CASES:
        plan, f = _check_case_features(case, B200_SMS)
        seen[case.mode] |= f
        if plan.fast:
            pairs[case.mode] |= {(plan.P, s) for _, _, s in plan.launches}
            if len(plan.n_iters) == 1:
                iters |= plan.n_iters
            kc_split |= case.kc and plan.ct_splits > 1
    for mode in (0, 1):
        missing = [(p, s) for p in (1, 2, 4, 8) for s in range(8) if (p, s) not in pairs[mode]]
        assert not missing, f"MODE {mode}: no case for (P, S) in {missing}"
        need = {"xb1", "xb2", "spill", "early_return", "lane31", "a0_neg", "split", "uneven", "padded",
                "Pclamp", "generic", "clamp32768"}
        assert need <= seen[mode], f"MODE {mode} misses {sorted(need - seen[mode])}"
    assert {"u1", "u2", "u4"} <= seen[0]
    for variant, stages in STAGES.items():
        want = {1, stages - 1, stages, stages + 1}
        assert want <= iters, f"variant {variant}: no uniform per-CTA loop of {sorted(want - iters)} tiles"
    assert kc_split


# --------------------------------------------------------------------------------- helpers
def dev(a, device):
    return torch.from_numpy(np.ascontiguousarray(a)).to(device)


def dev_at(a, device, off):
    """Device copy of `a` starting `off` elements into a fresh allocation (off = 0: aligned)."""
    t = torch.from_numpy(np.ascontiguousarray(a))
    flat = torch.empty(t.numel() + 16, dtype=t.dtype, device=device)
    out = flat[off:off + t.numel()].view(t.shape)
    out.copy_(t.to(device))
    return out


_TORCH = {"uint8": torch.uint8, "uint16": torch.uint16, "float32": torch.float32, "float64": torch.float64}


def out_buffer(image_shape, dtype, layout, device):
    """A sentinel-filled byte buffer holding a (C,T,Him,Wim) image of the given layout with 256
    guard bytes after it and 16 or more before it.  Returns (buffer, image view, pitch, front)."""
    c, t, him, wim = image_shape
    itemsize = np.dtype(dtype).itemsize
    pitch, front = _layout(layout, wim, itemsize)
    n = c * t * him * pitch * itemsize
    raw = torch.full((front + n + 256,), SENTINEL, dtype=torch.uint8, device=device)
    image = raw[front:front + n].view(_TORCH[dtype]).view(c, t, him, pitch)[..., :wim]
    return raw, image, pitch, front


def check_raw(raw, front, pitch, want, msg):
    """The visible image equals `want`; every other byte of the buffer (row padding, guards)
    still holds the sentinel."""
    got = raw.cpu().numpy()
    c, t, him, wim = want.shape
    n = c * t * him * pitch * want.itemsize
    vis = got[front:front + n].view(want.dtype).reshape(c, t, him, pitch)[..., :wim]
    np.testing.assert_array_equal(vis, want, err_msg=msg)
    exp = np.full_like(got, SENTINEL)
    exp[front:front + n].view(want.dtype).reshape(c, t, him, pitch)[..., :wim] = want
    bad = np.flatnonzero(got != exp)
    assert bad.size == 0, (f"{msg}: {bad.size} bytes outside the image were written, first at byte "
                           f"{bad[0] - front} of the image (pitch {pitch * want.itemsize} bytes)")


def _tiles(rng, dtype, shape):
    if dtype == "uint16":
        return rng.integers(0, 65535, shape, dtype=np.uint16, endpoint=True)
    if dtype == "uint8":
        return rng.integers(0, 255, shape, dtype=np.uint8, endpoint=True)
    return (rng.standard_normal(shape) * 1000).astype(dtype)


def _ff_data(rng, shape, per_channel):
    """uint16 tiles with clipped and saturated pixels, smooth flat in [0.65, 1.35] and dark
    around 100; per channel (K = C) every channel gets tables of its own."""
    c, t, r, cc, h, w = shape
    tiles = np.clip(rng.normal(3000, 1500, shape), 0, 65535).astype(np.uint16)
    low = rng.random(shape) < 0.05
    tiles[low] = rng.integers(0, 90, int(low.sum()))      # below dark -> 0
    tiles.reshape(-1)[rng.integers(0, tiles.size)] = 65535
    yy, xx = np.mgrid[0:h, 0:w]
    flat = 1.0 + 0.35 * np.cos(yy / h * 2.1 + 0.2) * np.sin(xx / max(w, 1) * 1.7 + 0.3)
    dark = 100.0 + 5.0 * np.sin(yy * 0.37 + xx * 0.11)
    if per_channel:
        flat = np.stack([flat * (1 + 0.13 * k) for k in range(c)])[:, None, None, None]
        dark = np.stack([dark + 7 * k for k in range(c)])[:, None, None, None]
    return tiles, flat, dark


@pytest.fixture(params=sorted(STAGES), ids=[f"v{v}-{STAGES[v]}st" for v in sorted(STAGES)])
def stitch_variant(request, cuda_device):
    """Runs the test under one stitch variant and restores the previous one afterwards."""
    from magnify_b200 import _lib

    lib = _lib.load()
    old = lib.mgb_set_stitch_variant(request.param)
    try:
        yield request.param
    finally:
        lib.mgb_set_stitch_variant(old)


def _set_iters(monkeypatch, iters):
    if iters is None:
        monkeypatch.delenv("MGB_STITCH_ITERS", raising=False)
    else:
        monkeypatch.setenv("MGB_STITCH_ITERS", str(iters))


def _direct_flatfield(tiles_d, image, pitch, shape, overlap, plan):
    """Pass 1, the coefficient tables and mgb_flatfield_stitch_u16 called directly; returns rc."""
    from magnify_b200 import _lib, ops

    c, t, r, cc, h, w = shape
    ops.flatfield_maxima(tiles_d, plan)
    _lib.call("mgb_flatfield_tables", ops._ptr(plan.flat), ops._ptr(plan.dark), plan.k, h * w, ops._ptr(plan.maxima),
              ops._ptr(plan.gain), ops._ptr(plan.bias), ops._stream())
    return _lib.try_call("mgb_flatfield_stitch_u16", ops._ptr(tiles_d), ops._ptr(image), pitch, c, t, r, cc, h, w,
                         overlap, plan.k, ops._ptr(plan.flat), ops._ptr(plan.dark), ops._ptr(plan.gain),
                         ops._ptr(plan.bias), ops._ptr(plan.maxima), ops._stream())


# ------------------------------------------------------------------------------ the matrix
@gpu
@pytest.mark.parametrize("case", CASES, ids=[_case_id(c) for c in CASES])
def test_stitch_configuration(cuda_device, stitch_variant, monkeypatch, case):
    from magnify_b200 import _lib, ops

    plan, _ = _check_case_features(case, ops.sm_count())
    _set_iters(monkeypatch, case.iters)
    rng = np.random.default_rng(CASES.index(case))
    c, t, r, cc, h, w = case.shape
    image_shape = ops.stitched_shape(case.shape, case.overlap)
    msg = f"{_case_id(case)} variant {stitch_variant}"

    if case.mode == 0:
        tiles = _tiles(rng, case.dtype, case.shape)
        want = o_st.stitch(tiles, case.overlap)
        tiles_d = dev_at(tiles, cuda_device, case.toff)
        raw, image, pitch, front = out_buffer(image_shape, case.dtype, case.layout, cuda_device)
        used = ctypes.c_int(-1)
        with torch.cuda.device(cuda_device):
            _lib.call("mgb_stitch", ops._ptr(tiles_d), ops._ptr(image), pitch, c, t, r, cc, h, w, case.overlap,
                      tiles.itemsize, ctypes.byref(used), ops._stream())
        assert used.value == int(plan.fast), msg
        check_raw(raw, front, pitch, want, msg)
        raw2, image2, _, _ = out_buffer(image_shape, case.dtype, case.layout, cuda_device)
        assert ops.stitch(tiles_d, case.overlap, out=image2).data_ptr() == image2.data_ptr()
        assert torch.equal(raw2, raw), msg
        return

    tiles, flat, dark = _ff_data(rng, case.shape, case.kc)
    want = o_st.stitch(o_ff.flatfield_correct(tiles, flat, dark), case.overlap)
    tiles_d = dev_at(tiles, cuda_device, case.toff)
    raw, image, pitch, front = out_buffer(image_shape, "uint16", case.layout, cuda_device)
    ffp = ops.FlatFieldPlan(case.shape, flat, dark, device=cuda_device)
    assert ffp.k == (c if case.kc else 1)
    with torch.cuda.device(cuda_device):
        rc = _direct_flatfield(tiles_d, image, pitch, case.shape, case.overlap, ffp)
    assert rc == (0 if plan.fast else _lib.MGB_EALIGN), msg
    assert tuple(ffp.maxima.cpu().numpy()) == o_ff.flatfield_maxima(tiles, flat, dark), msg
    if rc == 0:
        check_raw(raw, front, pitch, want, msg)
    else:
        assert bool((raw == SENTINEL).all()), f"{msg}: MGB_EALIGN after writing the image"
    raw2, image2, _, _ = out_buffer(image_shape, "uint16", case.layout, cuda_device)
    ops.flatfield_stitch(tiles_d, overlap=case.overlap, plan=ops.FlatFieldPlan(case.shape, flat, dark, device=cuda_device),
                         out=image2)
    check_raw(raw2, front, pitch, want, msg + " (ops.flatfield_stitch)")
    if rc == 0:
        assert torch.equal(raw2, raw), msg


# ------------------------------------------------- exact recompute next to the fast path
@gpu
@pytest.mark.parametrize("col", range(8))
def test_flatfield_exact_pixel_in_fast_vector(cuda_device, stitch_variant, col):
    """flat = 1 with an integer dark at tile columns x with (x - clip) % 8 == col, flat in (1, 1.5]
    elsewhere, and the brightest pixel on such a column (so M2 == M): those pixels land exactly
    on integers and force the whole-vector exact recompute; the other 7 pixels of the vector must
    still match.  Every 4th row also has a rejected gain (flat = 0.04, gain > 16) at (x - clip) %
    8 == col + 3, whose fast-path value is 0.  With w = 265 and Cc = 8 the eight phase slices put
    the column at every lane of the output vector, each with its own input shift S: over col =
    0..7 every (lane, S) pair occurs."""
    from magnify_b200 import ops

    shape, overlap = (1, 2, 2, 8, 12, 272), 7
    c, t, r, cc, h, w = shape
    clip = overlap // 2
    plan = stitch_plan(shape, overlap, 2, 1, ops.sm_count(), TARGET_ITERS[1])
    assert plan.P == 8 and {s for _, _, s in plan.launches} == set(range(8))
    rng = np.random.default_rng(100 + col)
    xs = np.arange(w)
    exact_cols = xs[(xs - clip) % 8 == col]
    reject_cols = xs[(xs - clip) % 8 == (col + 3) % 8]
    flat = 1.5 - 0.5 * rng.random((h, w))
    dark = rng.uniform(20, 200, (h, w))
    flat[:, exact_cols] = 1.0
    dark[:, exact_cols] = rng.integers(20, 200, (h, exact_cols.size))
    tiles = np.clip(rng.normal(3000, 1500, shape), 0, 60000).astype(np.uint16)
    rej_rows = np.arange(1, h, 4)
    flat[np.ix_(rej_rows, reject_cols)] = 0.04
    small = np.ceil(dark[np.ix_(rej_rows, reject_cols)]) + rng.integers(1, 50, (t, r, cc, rej_rows.size, reject_cols.size))
    tiles[0][np.ix_(range(t), range(r), range(cc), rej_rows, reject_cols)] = small.astype(np.uint16)
    y0, x0 = 5, exact_cols[7]
    dark[y0, x0] = 0.0
    tiles[0, 1, 1, 3, y0, x0] = 65535
    m, m2 = o_ff.flatfield_maxima(tiles, flat, dark)
    assert m == m2 == 65535.0
    want = o_st.stitch(o_ff.flatfield_correct(tiles, flat, dark), overlap)
    image_shape = want.shape
    raw, image, pitch, front = out_buffer(image_shape, "uint16", "alloc", cuda_device)
    ffp = ops.FlatFieldPlan(shape, flat, dark, device=cuda_device)
    with torch.cuda.device(cuda_device):
        assert _direct_flatfield(dev(tiles, cuda_device), image, pitch, shape, overlap, ffp) == 0
    gain = ffp.gain.cpu().numpy()[0]
    assert (gain[np.ix_(rej_rows, reject_cols)] == 0).all() and (gain[:, exact_cols] == 1).all()
    check_raw(raw, front, pitch, want, f"col {col}")


# -------------------------------------------------------------------------- maxima, pass 1
def tilemax_splits(n_planes, hw, K, sm_count):
    """The split of the uint16 maxima pass over planes (ops._maxima_pass restated)."""
    base = -(-(hw // 8) // 256) * K
    return max(1, min(n_planes // 8 if n_planes >= 16 else 1, -(-sm_count * 16 // base), 4096))


def _oracle_maxima(tiles, flat, dark):
    """oracle.flatfield_maxima; a large stack is first reduced to its per-position maxima over
    the planes that share a table, which leaves both maxima unchanged: clip(x - dark, 0) and
    its quotient by flat > 0 are non-decreasing in x, IEEE rounding included."""
    if tiles.size <= 1 << 22:
        return o_ff.flatfield_maxima(tiles, flat, dark)
    c = tiles.shape[0]
    if np.ndim(flat) == 6:
        red = tiles.reshape(c, -1, *tiles.shape[-2:]).max(1)
        return o_ff.flatfield_maxima(red, flat[:, 0, 0, 0], dark[:, 0, 0, 0] if np.ndim(dark) == 6 else dark)
    return o_ff.flatfield_maxima(tiles.reshape(-1, *tiles.shape[-2:]).max(0), flat, dark)


def _maxima_tables(rng, c, h, w, per_channel):
    flat = rng.uniform(0.8, 1.2, (h, w))
    dark = rng.uniform(90, 110, (h, w))
    if per_channel:
        flat = np.stack([flat * (1 + 0.05 * k) for k in range(c)])[:, None, None, None]
        dark = np.stack([dark + 2 * k for k in range(c)])[:, None, None, None]
    return flat, dark


@gpu
@pytest.mark.parametrize("where", ["first", "last"])
@pytest.mark.parametrize("regime,per_channel", [("one", False), ("one", True), ("eighth", False), ("eighth", True),
                                                ("cap", False)])
def test_tilemax_maxima(cuda_device, regime, per_channel, where):
    """The uint16 maxima pass (per-position maxima split over planes, then M and M2) bit for bit
    against the oracle, with the brightest pixel alone in the first or the last plane of a split:
    one split (fewer than 16 planes), n_planes // 8 splits, and the 16 x SMs cap."""
    from magnify_b200 import ops

    sms = ops.sm_count()
    c = 3 if per_channel else 1 if regime == "one" else 2
    if regime == "one":
        c, t, r, cc, h, w = c, 2, 2, 3, 32, 64
    elif regime == "eighth":
        c, t, r, cc, h, w = c, 5, 2, 4, 64, 64
    else:   # enough 512 x 512 planes that n_planes // 8 exceeds the cap
        cap = -(-sms * 16 // 128)
        c, t, r, cc, h, w = 1, 8 * (cap + 1), 1, 1, 512, 512
    shape = (c, t, r, cc, h, w)
    k = c if per_channel else 1
    n_planes = t * r * cc * (1 if per_channel else c)
    splits = tilemax_splits(n_planes, h * w, k, sms)
    if regime == "one":
        assert n_planes < 16 and splits == 1
    elif regime == "eighth":
        assert splits == n_planes // 8 > 1
    else:
        assert 1 < splits == -(-sms * 16 // (h * w // 2048)) < n_planes // 8
    rng = np.random.default_rng([len(regime), per_channel, where == "first"])
    tiles = rng.integers(0, 60000, shape, dtype=np.uint16)
    s = splits // 2 if splits > 1 else 0
    plane = n_planes * s // splits if where == "first" else n_planes * (s + 1) // splits - 1
    table_planes = tiles.reshape(k, n_planes, h, w)
    table_planes[k - 1, plane, h // 3, w // 5] = 65535
    flat, dark = _maxima_tables(rng, c, h, w, per_channel)
    plan = ops.FlatFieldPlan(shape, flat, dark, device=cuda_device)
    got = tuple(ops.flatfield_maxima(dev(tiles, cuda_device), plan).cpu().numpy())
    want = _oracle_maxima(tiles, flat, dark)
    assert want[0] == 65535 - dark.reshape(-1, h, w)[k - 1, h // 3, w // 5]
    assert got == want


@gpu
@pytest.mark.parametrize("kind", ["uint8", "float32", "float64", "uint16-hw-odd", "uint16-misaligned"])
@pytest.mark.parametrize("per_channel", [False, True], ids=["K1", "KC"])
def test_generic_maxima(cuda_device, kind, per_channel):
    """The element-wise maxima pass (any dtype, H * W % 8 != 0, a misaligned tile pointer)
    bit for bit against the oracle."""
    from magnify_b200 import ops

    rng = np.random.default_rng(7 + len(kind) + per_channel)
    h, w = (15, 15) if kind == "uint16-hw-odd" else (16, 24)
    shape = (3, 2, 2, 2, h, w)
    dtype = kind.split("-")[0]
    tiles = _tiles(rng, dtype, shape)
    if dtype.startswith("float"):
        tiles = np.abs(tiles) * 3 - 500     # some pixels below dark
    tiles_d = dev_at(tiles, cuda_device, 1 if kind.endswith("misaligned") else 0)
    assert (tiles_d.data_ptr() % 16 != 0) == kind.endswith("misaligned")
    flat, dark = _maxima_tables(rng, shape[0], h, w, per_channel)
    plan = ops.FlatFieldPlan(shape, flat, dark, device=cuda_device)
    got = tuple(ops.flatfield_maxima(tiles_d, plan).cpu().numpy())
    assert got == o_ff.flatfield_maxima(tiles, flat, dark)


@gpu
@pytest.mark.parametrize("dtype", ["uint16", "float32"])
@pytest.mark.parametrize("per_channel", [False, True], ids=["K1", "KC"])
def test_maxima_accumulate_blocks(cuda_device, dtype, per_channel):
    """flatfield_maxima_accumulate over every (channel, timepoint) block into a zeroed
    plan.maxima equals the maxima of the whole stack (18 planes per block: a split pass)."""
    from magnify_b200 import ops

    rng = np.random.default_rng(11 + per_channel)
    shape = (3, 4, 2, 9, 16, 24)
    c, t = shape[:2]
    tiles = rng.integers(0, 60000, shape, dtype=np.uint16)
    tiles[2, 3, 1, 0, 4, 7] = 65535           # first plane of the second split of the last block
    tiles = tiles.astype(dtype)
    flat, dark = _maxima_tables(rng, c, 16, 24, per_channel)
    plan = ops.FlatFieldPlan(shape, flat, dark, device=cuda_device)
    tiles_d = dev(tiles, cuda_device)
    plan.maxima.zero_()
    for ci in range(c):
        for ti in range(t):
            ops.flatfield_maxima_accumulate(tiles_d[ci, ti], plan, ci)
    want = o_ff.flatfield_maxima(tiles, flat, dark)
    assert tuple(plan.maxima.cpu().numpy()) == want
    assert tuple(ops.flatfield_maxima(tiles_d, plan).cpu().numpy()) == want


@gpu
@pytest.mark.parametrize("per_channel", [False, True], ids=["K1", "KC"])
def test_flatfield_stitch_given_maxima(cuda_device, stitch_variant, per_channel):
    """Maxima passed in as their own tensor (as after an all-reduce over ranks) are copied into
    plan.maxima and used as they are, not recomputed from the local tiles."""
    from magnify_b200 import ops

    rng = np.random.default_rng(21 + per_channel)
    shape, overlap = (2, 2, 2, 3, 16, 64), 6
    tiles, flat, dark = _ff_data(rng, shape, per_channel)
    m, m2 = o_ff.flatfield_maxima(tiles, flat, dark)
    given = (m * 1.0625, m2 * 1.375)
    want = o_st.stitch(o_ff.flatfield_correct(tiles, flat, dark, maxima=given), overlap)
    maxima = torch.tensor(given, dtype=torch.float64, device=cuda_device)
    plan = ops.FlatFieldPlan(shape, flat, dark, device=cuda_device)
    raw, image, pitch, front = out_buffer(want.shape, "uint16", "alloc", cuda_device)
    ops.flatfield_stitch(dev(tiles, cuda_device), overlap=overlap, plan=plan, maxima=maxima, out=image)
    check_raw(raw, front, pitch, want, "given maxima")
    assert tuple(plan.maxima.cpu().numpy()) == given and tuple(maxima.cpu().numpy()) == given


@gpu
@pytest.mark.parametrize("w,features", [(264, {"P1"}), (2056, {"P1", "xb2", "spill"}), (265, {"generic"})],
                         ids=["w264", "w2056", "w265"])
def test_flatfield_correct_tile_layout(cuda_device, w, features):
    """flatfield_correct runs each tile as its own 1 x 1 image at overlap 0: a row of 33
    vectors (lane 31 of the second warp), a row of 257 vectors (two x-blocks) and an odd width
    (MGB_EALIGN -> exact generic kernel)."""
    from magnify_b200 import ops

    rng = np.random.default_rng(w)
    shape = (2, 2, 1, 2, 6, w)
    c, t, r, cc, h, _ = shape
    plan = stitch_plan((c, t * r * cc, 1, 1, h, w), 0, 2, 1, ops.sm_count(), TARGET_ITERS[1])
    assert features <= plan_features(plan, w, w)
    tiles, flat, dark = _ff_data(rng, shape, True)
    got = ops.flatfield_correct(dev(tiles, cuda_device), flat, dark)
    np.testing.assert_array_equal(got.cpu().numpy(), o_ff.flatfield_correct(tiles, flat, dark))
