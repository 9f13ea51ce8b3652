"""Every configuration of the staged and plain ROI gather and of the standalone reductions
against the float64 oracle.

Without the fused list kernels (`test_gpu_gather_fused.py`), a gather call takes the staged
kernels of roi_tma.cu -- a window staged in shared memory by TMA or cp.async and re-aligned by
a vector, word or element copy loop unrolled for 12, 21 or 36 vectors per lane (or a run-time
loop), 8 or 4 warps of 2 to 4 stages, one CTA per marker or, for many markers with quad rows,
one warp per marker with 12, 20 or 24 quads per lane -- or the plain word / element kernels of
roi.cu.  `staged_plan` restates the host logic that picks one of them; each case of the matrix
names the features it is meant to reach, asserts the launch `ops.last_gather_path()` reports
against the plan, and compares crops (bit for bit), counts and sums (exactly), means (1e-12
relative) and the medians of the separate exact-median pass with `oracle.rois.gather_rois` /
`oracle.reduce`.  Crops go into a buffer whose guard bytes before and after must survive.

The standalone reductions follow: `roi_median` at both sides of every keys-per-thread class of
its kernels (uint16 and float32, with ties, signed zeros, infinities, NaN, subnormals and
float32 overflow), `roi_stats` of uint16 crops on the word and element kernels, and of float32
crops.

`test_matrix_covers_every_configuration` needs no GPU: from the case list and `staged_plan` at
the shared-memory limits of a B200 it checks that every class above is reached.
"""
import ctypes
import itertools
from collections import namedtuple

import numpy as np
import pytest
import torch

import test_gpu_gather_fused as fused
from oracle import reduce as o_red
from oracle import rois as o_rois

gpu = pytest.mark.gpu

# B200: shared memory per block (opt-in), shared memory per SM, SMs
B200_LIMITS = (232448, 233472, 148)
TMA_MAX_WARPS = 8
PLAIN_WARPS = 8          # kThreads / 32 of the plain kernels
WPM_MIN_MARKERS = 2048
GUARD = 64               # guard bytes before and after every crop buffer
SENTINEL = 0xA5

Path = namedtuple("Path", "kernel unroll copy_loop warps stages loader stats store")


# ------------------------------------------------------------------------------ launch plan
def copy_loop(L, wu, roi_align, quads):
    """roi_stage.cuh copy_loop: roi_align = largest power of two (up to 16) dividing the crop
    buffer's byte address, None for summaries only (which counts as aligned)."""
    a = 16 if roi_align is None else roi_align
    if wu % 8 == 0 and wu > 8 and a >= 16:
        return "vector"
    if quads and wu % 2 == 0 and (L * wu) % 4 == 0 and a >= 8 and (L * wu // 4 + 31) // 32 <= 24:
        return "quad"
    if wu % 2 == 0 and wu > 2 and a >= 4:
        return "word"
    return "element"


def _vpl_class(v):
    return 12 if 0 < v <= 12 else 21 if 12 < v <= 21 else 36 if 21 < v <= 36 else 0


def staged_plan(L, itemsize, C, T, M, stats=False, store=True, roi_align=16, image_align=16, pitch_bytes=None,
                mask_align=16, loader=0, warps=None, tma=True, limits=B200_LIMITS):
    """The launch of gather_common restated, for calls that do not take the fused list kernels
    (`roi_gather`, or summaries with unknown or too large mask counts): the staged window set-up
    (stage_window), the warp and stage search and the warp-per-marker choice of roi_gather_tma,
    then the plain word / element kernels.  image_align: largest power of two (up to 16) dividing
    the image's byte address; pitch_bytes: its row pitch; loader: mgb_set_gather_loader's value;
    warps: MGB_GATHER_WARPS (None: unset)."""
    max_smem = limits[0]
    pitch_bytes = L * itemsize if pitch_bytes is None else pitch_bytes
    unit = itemsize // 2
    if tma and itemsize >= 2 and pitch_bytes % 16 == 0 and image_align >= 16:
        wu = L * unit
        wpu = (wu + 14) & ~7
        if wpu <= 256 and L <= 256:
            loop = copy_loop(L, wu, roi_align, False)
            stage = (L * wpu * 2 + 127) & ~127
            mask_bytes = 2 * ((L * wu + 15) & ~15) if stats else 0
            fixed = mask_bytes + TMA_MAX_WARPS * 8 * 8 + T * 4 + 128
            budget = max_smem - fixed - 1024 if max_smem > fixed + 1024 else 0
            nw = 4 if warps == 4 else TMA_MAX_WARPS
            ns = budget // (nw * stage)
            if ns < 2:
                nw = 4
                ns = budget // (nw * stage)
            ns = min(ns, 4)
            if ns >= 2:
                masks_words = not stats or (L * L % 4 == 0 and mask_align >= 4)
                if (not loader & 2 and unit == 1 and copy_loop(L, wu, roi_align, True) == "quad"
                        and M >= WPM_MIN_MARKERS and masks_words):
                    fixed_w = TMA_MAX_WARPS * 8 * 8 + T * 4 + 128
                    budget_w = max_smem - fixed_w - 1024 if max_smem > fixed_w + 1024 else 0
                    ns_w = min(budget_w // (TMA_MAX_WARPS * stage), 4)
                    if ns_w >= 2:
                        q = ((L * wu) // 4 + 31) // 32
                        return Path("staged-wpm", 12 if q <= 12 else 20 if q <= 20 else 24, "quad", TMA_MAX_WARPS,
                                    ns_w, "tma", stats, store)
                vpl = (L * (wu // 8) + 31) // 32 if loop == "vector" else 0
                return Path("staged-cta", _vpl_class(vpl), loop, nw, ns, "cp.async" if loader & 1 else "tma",
                            stats, store)
    lu = L * max(unit, 1)
    words = (itemsize >= 2 and lu % 2 == 0 and lu > 2 and image_align >= 4 and (not store or roi_align >= 4)
             and (not stats or mask_align >= 2))
    return Path("plain-words" if words else "plain-scalar", 0, "word" if words else "element", PLAIN_WARPS, 0, None,
                stats, store)


def path_features(path):
    f = {path.kernel, f"{path.kernel}:u{path.unroll}", f"{path.kernel}:{path.copy_loop}",
         f"ST{int(path.stats)}{int(path.store)}", f"{path.kernel}:ST{int(path.stats)}{int(path.store)}"}
    if path.kernel.startswith("staged"):
        f |= {f"w{path.warps}", f"s{path.stages}", f"w{path.warps}s{path.stages}", f"loader:{path.loader}"}
    return f


# ---------------------------------------------------------------------------- case matrix
Case = namedtuple("Case", "dtype L C T M call tmk order loader warps layout roi_off mask_off tma values features")
# call: "gather" (ops.roi_gather), "stats" / "stats_noroi" (mgb_roi_gather_stats_u16 with unknown
# mask counts, crops stored or not), "ops_stats" / "ops_stats_noroi" (ops.roi_gather_stats with
# masks over the list capacities).  layout: "alloc" (ops.alloc_image, padded pitch unless W is
# aligned), "dense" (W a multiple of 16 bytes), "off1" / "off2" (dense image 1 / 2 elements into
# its buffer), "pitch_odd" (pitch of W + 1 elements).  roi_off / mask_off: byte offsets of the crop
# buffer / both masks in their allocations.

MASK_T = {"gap": fused.MASK_T["gap"], "unsorted": fused.MASK_T["unsorted"]}   # T = 4; "gap": a mask timestep owns no timepoint
for _t in (33, 64, 65):
    MASK_T[f"t{_t}"] = (3, [(7 * i) % 3 for i in range(_t)])


def mask_timesteps(key, T):
    """(Tm, mask_t) of a case: "one" (Tm = 1), "all" (Tm = T) or one of MASK_T."""
    if key == "one":
        return 1, [0] * T
    if key == "all":
        return T, list(range(T))
    assert len(MASK_T[key][1]) == T, (key, T)
    return MASK_T[key]


def _case(dtype="uint16", L=40, C=2, T=4, M=12, call="gather", tmk="one", order=False, loader=0, warps=None,
          layout="alloc", roi_off=0, mask_off=0, tma=True, values="random", features=()):
    return Case(dtype, L, C, T, M, call, tmk, order, loader, warps, layout, roi_off, mask_off, tma, values,
                frozenset(features))


def _largest_staged(itemsize, stats, T=2, limits=B200_LIMITS):
    return max(L for L in range(1, 257)
               if staged_plan(L, itemsize, 1, T, 12, stats, pitch_bytes=16 * 64, limits=limits).kernel == "staged-cta")


L_MAX_U16 = _largest_staged(2, False)
L_MAX_U16_STATS = _largest_staged(2, True)
L_MAX_F32 = _largest_staged(4, False)
L_MAX_F64 = _largest_staged(8, False)

CASES = [
    # staged CTA kernel, uint16: every unroll class with crops, with summaries, summaries only
    _case(L=16, features={"staged-cta:u12", "staged-cta:vector", "w8s4"}),
    _case(L=40, call="stats", tmk="all", order=True, features={"staged-cta:u12", "staged-cta:ST11"}),
    _case(L=56, call="stats_noroi", tmk="gap", features={"staged-cta:u21", "staged-cta:ST10"}),
    _case(L=72, tmk="unsorted", order=True, features={"staged-cta:u21", "staged-cta:ST01"}),
    _case(L=80, call="stats", features={"staged-cta:u36", "w4s3"}),
    _case(L=96, order=True, features={"staged-cta:u36"}),
    _case(L=104, call="stats", tmk="all", features={"staged-cta:u0", "staged-cta:vector"}),
    _case(L=112, C=1, T=2, M=5, features={"staged-cta:u0", "staged-cta:vector", "w4s2"}),
    _case(L=L_MAX_U16, C=1, T=2, M=5, features={"staged-cta:element", "w4s2"}),
    _case(L=128, C=1, T=2, M=6, features={"plain-words:ST01"}),   # 4 warps x 2 stages do not fit
    # the largest window with summaries, all pixels 65535 under full 0/255 masks: 32-bit warp sums
    _case(L=L_MAX_U16_STATS, C=1, T=2, M=5, call="stats", values="saturated", features={"staged-cta:ST11", "w4s2"}),
    # word and element loops
    _case(L=34, features={"staged-cta:word"}),
    _case(L=50, call="stats", tmk="unsorted", features={"staged-cta:word", "staged-cta:ST11"}),
    _case(L=48, roi_off=4, features={"staged-cta:word"}),
    _case(L=48, roi_off=8, call="stats", features={"staged-cta:word"}),
    _case(L=33, call="stats", tmk="gap", order=True, features={"staged-cta:element"}),
    _case(L=1, features={"staged-cta:element"}),
    _case(L=2, call="stats", features={"staged-cta:element"}),
    _case(L=40, roi_off=2, features={"staged-cta:element"}),
    _case(L=8, call="stats_noroi", features={"staged-cta:word"}),   # rows of a single vector
    # stage counts and warps near the thresholds
    _case(L=64, call="stats", features={"w8s3"}),
    _case(L=72, call="stats", features={"w8s2"}),
    _case(L=88, features={"w4s3"}),
    _case(L=48, warps=4, call="stats", features={"w4s4"}),
    _case(L=96, warps=4, features={"w4"}),
    # cp.async loader, windows at the right edge of padded and dense images
    _case(L=40, loader=1, call="stats", layout="dense", features={"loader:cp.async"}),
    _case(L=72, loader=1, layout="alloc", order=True, features={"loader:cp.async", "staged-cta:u21"}),
    _case(L=34, loader=1, call="stats_noroi", tmk="all", layout="alloc", features={"loader:cp.async"}),
    _case(L=33, loader=1, layout="dense", features={"loader:cp.async", "staged-cta:element"}),
    _case(L=104, loader=1, call="stats", features={"loader:cp.async", "w4"}),
    # more than 32 timepoints: list_timepoints loops over several ballots
    _case(L=24, C=1, T=33, M=5, call="stats", tmk="t33", features={"staged-cta:ST11"}),
    _case(L=24, C=1, T=64, M=4, call="stats", tmk="t64", order=True, loader=1, features={"loader:cp.async"}),
    _case(L=34, C=1, T=65, M=4, call="stats_noroi", tmk="t65", features={"staged-cta:ST10"}),
    _case(L=16, C=1, T=65, M=3, features={"staged-cta:ST01"}),
    # roi_gather_stats itself with masks over the list capacities (bg > 2560 pixels)
    _case(L=56, call="ops_stats", tmk="all", features={"staged-cta:ST11"}),
    _case(L=64, call="ops_stats_noroi", order=True, features={"staged-cta:ST10"}),
    # float32 and float64 crops (2 and 4 units per element)
    _case("float32", L=8, features={"staged-cta:vector", "staged-cta:u12"}),
    _case("float32", L=4, features={"staged-cta:word"}),
    _case("float32", L=17, order=True, features={"staged-cta:word"}),
    _case("float32", L=20, roi_off=4, features={"staged-cta:word"}),
    _case("float32", L=1, features={"staged-cta:element"}),
    _case("float32", L=60, features={"staged-cta:u36"}),
    _case("float32", L=L_MAX_F32, C=1, T=2, M=4, loader=1, features={"staged-cta:u0"}),
    _case("float32", L=L_MAX_F32 + 1, C=1, T=2, M=4, features={"plain-words"}),
    _case("float64", L=2, features={"staged-cta:word"}),
    _case("float64", L=3, features={"staged-cta:word"}),
    _case("float64", L=8, tmk="all", features={"staged-cta:vector"}),
    _case("float64", L=L_MAX_F64, C=1, T=2, M=4, features={"staged-cta:u0"}),
    _case("float64", L=L_MAX_F64 + 1, C=1, T=2, M=4, features={"plain-words"}),
    _case("float64", L=63, C=1, T=2, M=3, features={"plain-words"}),
    # warp-per-marker kernel: 2048 markers or more, quad rows
    _case(L=38, C=1, T=2, M=2048, features={"staged-wpm:u12", "staged-wpm:ST01"}),
    _case(L=50, C=1, T=2, M=2049, call="stats", order=True, features={"staged-wpm:u20", "staged-wpm:ST11"}),
    _case(L=54, C=1, T=2, M=2048, call="stats_noroi", tmk="all", features={"staged-wpm:u24", "staged-wpm:ST10"}),
    _case(L=54, C=1, T=2, M=2050, features={"staged-wpm:u24"}),
    _case(L=50, C=1, T=2, M=2048, loader=1, features={"staged-wpm:u20"}),
    _case(L=38, C=1, T=2, M=2047, features={"staged-cta:word"}),
    _case(L=38, C=1, T=2, M=2048, call="stats", mask_off=2, features={"staged-cta:word"}),
    _case(L=50, C=1, T=2, M=2048, loader=2, features={"staged-cta:word"}),
    _case(L=50, C=1, T=2, M=2048, loader=3, call="stats", features={"staged-cta:word", "loader:cp.async"}),
    # plain kernels
    _case("uint8", L=17, features={"plain-scalar:ST01"}),
    _case("uint8", L=40, layout="dense", features={"plain-scalar:ST01"}),
    _case(L=40, call="stats", layout="off2", features={"plain-words:ST11"}),
    _case(L=40, layout="off1", features={"plain-scalar:ST01"}),
    _case(L=34, layout="pitch_odd", features={"plain-words:ST01"}),
    _case(L=33, call="stats", layout="pitch_odd", features={"plain-scalar:ST11"}),
    _case(L=40, call="stats", mask_off=1, layout="dense", features={"staged-cta:ST11"}),
    _case(L=40, call="stats", mask_off=1, tma=False, features={"plain-scalar:ST11"}),
    _case(L=260, C=1, T=2, M=3, features={"plain-words:ST01"}),
    _case(L=257, C=1, T=1, M=2, call="stats", features={"plain-scalar:ST11"}),
    _case(L=48, call="stats", tma=False, tmk="unsorted", features={"plain-words:ST11"}),
    _case(L=48, call="stats_noroi", tma=False, features={"plain-words:ST10"}),
    _case(L=35, call="stats_noroi", tma=False, features={"plain-scalar:ST10"}),
    _case("float32", L=20, tma=False, features={"plain-words:ST01"}),
    _case("float64", L=7, tma=False, layout="off1", features={"plain-words:ST01"}),
    _case(L=36, tma=False, layout="off2", roi_off=2, features={"plain-scalar:ST01"}),
]

REQUIRED = {
    "staged-cta:u12", "staged-cta:u21", "staged-cta:u36", "staged-cta:u0",
    "staged-cta:vector", "staged-cta:word", "staged-cta:element",
    "staged-cta:ST01", "staged-cta:ST11", "staged-cta:ST10",
    "staged-wpm:u12", "staged-wpm:u20", "staged-wpm:u24",
    "staged-wpm:ST01", "staged-wpm:ST11", "staged-wpm:ST10",
    "w8", "w4", "s2", "s3", "s4", "w8s2", "w8s3", "w8s4", "w4s2", "w4s3", "w4s4",
    "loader:tma", "loader:cp.async",
    "plain-words:ST01", "plain-words:ST11", "plain-words:ST10",
    "plain-scalar:ST01", "plain-scalar:ST11", "plain-scalar:ST10",
}


def _itemsize(case):
    return np.dtype(case.dtype).itemsize


def _geometry(case):
    """(H, W, pitch in elements, image byte alignment) of a case's image."""
    itemsize = _itemsize(case)
    q = 16 // itemsize
    h = case.L + 23
    w = max(case.L + 61, 2 * case.L + 5)
    if case.layout in ("dense", "off1", "off2"):
        w = -(-w // q) * q
    elif w % q == 0:
        w += 3 if q > 1 else 0
    pitch = {"alloc": -(-w // q) * q, "pitch_odd": w + 1 if (w + 1) % 2 else w + 2}.get(case.layout, w)
    return h, w, pitch, {"off1": itemsize, "off2": 2 * itemsize}.get(case.layout, 16)


def _stats(case):
    return case.call != "gather"


def _store(case):
    return not case.call.endswith("noroi")


def _align(off):
    return 16 if off % 16 == 0 else min(16, off & -off)


def case_plan(case, limits=B200_LIMITS):
    itemsize = _itemsize(case)
    h, w, pitch, image_align = _geometry(case)
    return staged_plan(case.L, itemsize, case.C, case.T, case.M, _stats(case), _store(case),
                       _align(case.roi_off) if _store(case) else None, image_align, pitch * itemsize,
                       _align(case.mask_off), case.loader, case.warps, case.tma, limits)


def _case_id(case):
    s = f"{case.dtype}-L{case.L}-{case.C}x{case.T}x{case.M}-{case.call}-{case.tmk}"
    for name in ("order", "loader", "warps", "roi_off", "mask_off"):
        if getattr(case, name):
            s += f"-{name}{int(getattr(case, name))}"
    if case.layout != "alloc":
        s += f"-{case.layout}"
    if not case.tma:
        s += "-notma"
    if case.values != "random":
        s += f"-{case.values}"
    return s


def test_matrix_covers_every_configuration():
    """No GPU: at the limits of a B200, every case reaches the features it names, and together
    they reach every kernel, unroll class, copy loop, warp x stage count, loader and
    summaries x crops combination of the staged and plain gather."""
    seen = set()
    for case in CASES:
        mask_timesteps(case.tmk, case.T)
        f = path_features(case_plan(case))
        missing = case.features - f
        assert not missing, f"{_case_id(case)} no longer reaches {sorted(missing)} (plan {case_plan(case)})"
        seen |= f
    assert not REQUIRED - seen, sorted(REQUIRED - seen)
    # the boundaries the matrix is built around
    assert staged_plan(38, 2, 1, 2, 2047, pitch_bytes=1024).kernel == "staged-cta"
    assert staged_plan(38, 2, 1, 2, 2048, pitch_bytes=1024).kernel == "staged-wpm"
    assert staged_plan(L_MAX_U16 + 1, 2, 1, 2, 5, pitch_bytes=1024).kernel == "plain-words"
    assert staged_plan(L_MAX_U16_STATS + 1, 2, 1, 2, 5, stats=True, pitch_bytes=1024).kernel == "plain-words"
    assert L_MAX_U16_STATS ** 2 * 65535 < 2 ** 32
    assert {c.T for c in CASES} >= {1, 2, 4, 33, 64, 65}
    assert len({_case_id(c) for c in CASES}) == len(CASES)


# ------------------------------------------------------------------------------ case data
def dev(a, device):
    return torch.from_numpy(np.ascontiguousarray(a)).to(device)


def _bits(a):
    """The raw bits of an array (bit-exact comparison of float crops, NaN included)."""
    a = np.ascontiguousarray(a)
    return a.view({1: np.uint8, 2: np.uint16, 4: np.uint32, 8: np.uint64}[a.itemsize])


def _image_values(case, rng, shape):
    itemsize = _itemsize(case)
    if case.values == "saturated":
        return np.full(shape, 65535, dtype=np.uint16)
    if case.dtype in ("float32", "float64"):   # any bit pattern: NaN, inf, subnormals, -0.0
        bits = rng.integers(0, 2 ** (8 * itemsize) - 1, shape, dtype=np.uint64, endpoint=True)
        return bits.astype({4: np.uint32, 8: np.uint64}[itemsize]).view(case.dtype)
    hi = np.iinfo(case.dtype).max
    image = rng.integers(0, hi, shape, dtype=case.dtype, endpoint=True)
    if shape[0] > 1:
        image[1] = np.clip(rng.normal(hi // 70, 30, image[1].shape), 0, hi).astype(case.dtype)   # many ties
    return image


def _markers(case, rng, h, w):
    """Centres (M, T) whose windows start at every left % 8 (and so at every residual shift of the
    staged window), at both image edges and at the right edge of the row."""
    L, M, T = case.L, case.M, case.T
    x = np.empty((M, T))
    y = np.empty((M, T))
    for i, t in itertools.product(range(M), range(T)):
        k = i * T + t
        s = k % 8
        left = s + 8 * int(rng.integers(0, (w - L - s) // 8 + 1))
        top = int(rng.integers(0, h - L + 1))
        x[i, t], y[i, t] = left + L // 2, top + L // 2
        if k % 11 == 9:
            x[i, t] = w + 4            # clipped to the right edge
        elif k % 13 == 12:
            x[i, t] = -3.0             # left edge
        if k % 6 == 5:
            y[i, t] = h + 2
    return x, y


def _device_image(case, image, device):
    itemsize = _itemsize(case)
    c, t, h, w = image.shape
    tdtype = {"uint8": torch.uint8, "uint16": torch.uint16, "float32": torch.float32, "float64": torch.float64}[case.dtype]
    host = torch.from_numpy(np.ascontiguousarray(image))
    if case.layout == "alloc":
        from magnify_b200 import ops

        out = ops.alloc_image(image.shape, tdtype, device)
    elif case.layout == "pitch_odd":
        _, _, pitch, _ = _geometry(case)
        out = torch.empty((c, t, h, pitch), dtype=tdtype, device=device)[..., :w]
    elif case.layout in ("off1", "off2"):
        off = 1 if case.layout == "off1" else 2
        out = torch.empty(image.size + 16, dtype=tdtype, device=device)[off:off + image.size].view(image.shape)
    else:
        out = torch.empty(image.shape, dtype=tdtype, device=device)
    out.copy_(host.to(device))
    _, _, pitch, align = _geometry(case)
    from magnify_b200 import ops

    assert ops.image_pitch(out) == pitch and out.data_ptr() % 16 == align % 16
    return out


def _guarded(shape, dtype, roi_off, device):
    """A contiguous output `roi_off` bytes past GUARD sentinel bytes, followed by GUARD more."""
    n = int(np.prod(shape)) * torch.empty(0, dtype=dtype).element_size()
    buf = torch.full((n + 2 * GUARD + 16,), SENTINEL, dtype=torch.uint8, device=device)
    start = GUARD + roi_off
    out = buf[start:start + n].view(dtype).view(shape)
    assert out.data_ptr() % 16 == roi_off % 16
    return buf, out, start, n


def _check_guards(buf, start, n, msg=""):
    b = buf.cpu().numpy()
    assert (b[:start] == SENTINEL).all() and (b[start + n:] == SENTINEL).all(), f"guard bytes overwritten {msg}"


def _masks(case, rng, tm):
    L, M = case.L, case.M
    if case.values == "saturated":
        full = np.ones((M, tm, L, L), dtype=bool)
        return full, full.copy()
    fg = rng.random((M, tm, L, L)) < rng.uniform(0.05, 0.6, (M, tm, 1, 1))
    bg = ~fg & (rng.random((M, tm, L, L)) < 0.8)
    if case.call.startswith("ops_stats"):
        bg[0, 0] = True                 # over the bg list capacity: not fused
        fg[0, 0] = False
    fg[min(1, M - 1)] = False           # an empty fg: NaN mean and median
    if M > 2:
        fg[2] = False
        fg[2, :, 0, L - 1] = True        # a single pixel
    return fg, bg


def _mask_bytes(case, rng, mask, device):
    """Device mask `case.mask_off` bytes into its buffer, with 255 (saturated) or random non-zero
    bytes where set."""
    vals = mask.astype(np.uint8) * (255 if case.values == "saturated" else rng.integers(1, 256, mask.shape))
    buf = torch.zeros(mask.size + 32, dtype=torch.uint8, device=device)
    view = buf[case.mask_off:case.mask_off + mask.size].view(mask.shape)
    view.copy_(dev(vals.astype(np.uint8), device))
    return view


def _stats_call(image, boxes, fg, bg, L, mask_t, tm, roi, order, device):
    """mgb_roi_gather_stats_u16 with unknown mask counts: the fused list kernels never apply."""
    from magnify_b200 import _lib, ops

    c, t, h, w = image.shape
    m = boxes.shape[0]
    stats = torch.empty((m, c, t, ops.NSTATS), dtype=torch.float64, device=device)
    done = ctypes.c_int(7)
    with torch.cuda.device(device):
        _lib.call("mgb_roi_gather_stats_u16", ops._ptr(image), ops.image_pitch(image), c, t, h, w, ops._ptr(boxes),
                  ops._ptr(order), ops._ptr(mask_t), tm, ops._ptr(fg), ops._ptr(bg), m, int(L), ops._ptr(roi),
                  ops._ptr(stats), 0, -1, -1, ctypes.byref(done), ops._stream())
    assert done.value == 0
    return stats


@pytest.fixture
def gather_settings(monkeypatch):
    """Restores the library's gather switches and the tuning variables after a test."""
    from magnify_b200 import _lib

    lib = _lib.load()
    for name in ("MGB_GATHER_WARPS", "MGB_GATHER_LAYOUT", "MGB_GATHER_SPLIT"):
        monkeypatch.delenv(name, raising=False)
    old_loader, old_tma = lib.mgb_set_gather_loader(0), lib.mgb_set_tma_enabled(1)
    yield lib
    lib.mgb_set_gather_loader(old_loader)
    lib.mgb_set_tma_enabled(old_tma)


def _run_case(case, seed, device, monkeypatch, lib):
    from magnify_b200 import ops

    rng = np.random.default_rng(seed)
    itemsize = _itemsize(case)
    h, w, _, _ = _geometry(case)
    image = _image_values(case, rng, (case.C, case.T, h, w))
    x, y = _markers(case, rng, h, w)
    tm, mask_t = mask_timesteps(case.tmk, case.T)
    mask_t = np.array(mask_t, dtype=np.int32)
    plan = case_plan(case, fused.device_limits(device))
    if case.warps:
        monkeypatch.setenv("MGB_GATHER_WARPS", str(case.warps))
    lib.mgb_set_gather_loader(case.loader)
    lib.mgb_set_tma_enabled(int(case.tma))

    image_d = _device_image(case, image, device)
    boxes = ops.bounding_boxes(dev(x, device), dev(y, device), case.L, w, h)
    lefts = boxes[..., 1].cpu().numpy()
    if plan.kernel.startswith("staged"):   # every residual shift the element size can produce
        unit = itemsize // 2
        assert set(((lefts * unit) & 7).ravel()) == set(range(0, 8, unit))
    order = dev(rng.permutation(case.M).astype(np.int32), device) if case.order else None
    want_roi = o_rois.gather_rois(image, x, y, case.L)
    shape = (case.M, case.C, case.T, case.L, case.L)
    tdtype = image_d.dtype
    buf = roi = None
    if _store(case):
        buf, roi, start, n = _guarded(shape, tdtype, case.roi_off, device)

    if case.call == "gather":
        got = ops.roi_gather(image_d, boxes, case.L, out=roi, order=order)
        assert got.data_ptr() == roi.data_ptr()
        assert ops.last_gather_path()[:8] == plan, _case_id(case)
        torch.cuda.synchronize(device)
        _check_guards(buf, start, n)
        np.testing.assert_array_equal(_bits(roi.cpu().numpy()), _bits(want_roi))
        return

    fg, bg = _masks(case, rng, tm)
    fg_d, bg_d = _mask_bytes(case, rng, fg, device), _mask_bytes(case, rng, bg, device)
    mask_t_d = dev(mask_t, device)
    if case.call.startswith("ops_stats"):
        counts = fused._counts(fg, bg)
        assert counts[1] > fused.BG_CAP
        roi_out, stats = ops.roi_gather_stats(image_d, boxes, fg_d, bg_d, case.L, mask_t=mask_t_d, want_roi=_store(case),
                                              out_roi=roi, order=order, medians=False, mask_counts=counts)
        assert roi_out is roi
    else:
        stats = _stats_call(image_d, boxes, fg_d, bg_d, case.L, mask_t_d, tm, roi, order, device)
    assert ops.last_gather_path()[:8] == plan, _case_id(case)
    want = o_red.masked_stats(want_roi, fg[:, mask_t], bg[:, mask_t])
    got = stats.cpu().numpy()
    assert np.isnan(got[..., 6:]).all()
    if roi is not None:
        torch.cuda.synchronize(device)
        _check_guards(buf, start, n)
        np.testing.assert_array_equal(roi.cpu().numpy(), want_roi)
        crops = roi
    else:
        crops = dev(want_roi, device)
    # the exact medians of the separate pass, into the stats records (stride 8)
    ops._median_into(crops, fg_d, mask_t_d, tm, stats, 6)
    ops._median_into(crops, bg_d, mask_t_d, tm, stats, 7)
    fused._check_stats(stats.cpu().numpy(), want, msg=_case_id(case))


@gpu
@pytest.mark.parametrize("case", CASES, ids=[_case_id(c) for c in CASES])
def test_staged_gather_configuration(cuda_device, monkeypatch, gather_settings, case):
    _run_case(case, CASES.index(case), cuda_device, monkeypatch, gather_settings)


# ------------------------------------------------------------------ standalone reductions
MEDIAN_LENGTHS = (1, 2, 32, 33, 50, 51, 73, 74, 101, 102, 128, 129, 160, 161, 200)


def median_npt(L):
    """Keys per thread of the median kernel launch_roi_median picks (0: the L > 160 kernel)."""
    npt = -(-L * L // 256)
    return next((n for n in (4, 10, 21, 40, 64, 100) if npt <= n), 0)


def test_median_lengths_cover_every_class():
    """No GPU: both sides of every keys-per-thread class edge."""
    classes = [median_npt(L) for L in MEDIAN_LENGTHS]
    assert set(classes) == {4, 10, 21, 40, 64, 100, 0}
    for edge in (32, 50, 73, 101, 128, 160):
        assert median_npt(edge) != median_npt(edge + 1), edge


# windows whose masks hold exactly 2 or 4 pixels with these values, one per (channel, time)
F32_SPECIAL = {
    2: [[1.0, 1.0 + 2.0 ** -23], [3e38, 3.2e38], [-0.0, 0.0], [-np.inf, np.inf], [np.nan, 5.0], [-2.5, 1e-45]],
    4: [[-0.0, 0.0, -0.0, 0.0], [-np.inf, -np.inf, 2.0, 3.0], [np.nan, -np.nan, 1e-40, 3e-40],
        [-3.0, -1.0, 2.0, 5.0], [-3e38, -3.3e38, -3.1e38, 1.0], [1e-45, 3e-45, -1e-45, 5e-45]],
}
U16_SPECIAL = {
    2: [[0, 65535], [65535, 65535], [0, 0], [1, 2], [65534, 65535], [7, 7]],
    4: [[0, 0, 65535, 65535], [0, 1, 65535, 65535], [3, 3, 3, 3], [65535, 65535, 65535, 0], [10, 11, 12, 13],
        [0, 65535, 1, 65534]],
}


def _median_case(dtype, L, rng):
    m, c, t, tm = 6, 2, 3, 2
    mask_t = np.array([1, 0, 1], dtype=np.int32)
    if dtype == np.float32:
        roi = (rng.standard_normal((m, c, t, L, L)) * 300).astype(np.float32)
        roi[0] = np.round(roi[0] / 50) * 50                                  # many ties
        nan_px = rng.random(roi.shape) < 0.05
        roi[nan_px] = np.where(rng.random(nan_px.sum()) < 0.5, np.float32(np.nan), -np.float32(np.nan))
        special = F32_SPECIAL
    else:
        roi = rng.integers(0, 65535, (m, c, t, L, L), dtype=np.uint16, endpoint=True)
        roi[0] = rng.integers(100, 104, roi[0].shape)                         # many ties
        roi[1, :, :, 0, 0] = 0
        roi[1, :, :, -1, -1] = 65535
        special = U16_SPECIAL
    mask = rng.random((m, tm, L, L)) < rng.uniform(0.2, 0.9, (m, tm, 1, 1))
    mask[1, 0, 0, 0] = mask[1, 0, -1, -1] = True
    mask[5] = False                                                          # empty: NaN
    if L * L >= 4:
        for mi, k in ((2, 2), (3, 4)):
            pos = rng.permutation(L * L)[:k]
            mask[mi] = False
            mask[mi].reshape(tm, -1)[:, pos] = True
            for w, (ci, ti) in enumerate(itertools.product(range(c), range(t))):
                roi[mi, ci, ti].reshape(-1)[pos] = np.array(special[k][w], dtype=roi.dtype)
    if L * L >= 2:
        mask[4] = False
        mask[4].reshape(tm, -1)[:, 0] = True                                 # one pixel
        mask[4, 1].reshape(-1)[1] = True                                     # and two
    return roi, mask, mask_t, tm


@gpu
@pytest.mark.parametrize("L", MEDIAN_LENGTHS)
@pytest.mark.parametrize("dtype", [np.uint16, np.float32], ids=["uint16", "float32"])
def test_roi_median_classes(cuda_device, dtype, L):
    """Exact masked medians at both sides of every keys-per-thread class, uint16 and float32,
    written with stride 8 into a stats buffer whose other columns must not change, against
    np.nanmedian of the roi in the dtype `roi.where(mask)` keeps (float32 middles averaged in
    float32: 1 and 1 + 2^-23 give 1, 3e38 and 3.2e38 give inf)."""
    from magnify_b200 import ops

    rng = np.random.default_rng(L * 3 + (dtype == np.float32))
    roi, mask, mask_t, tm = _median_case(dtype, L, rng)
    want = o_red.masked_median(roi, mask[:, mask_t])
    roi_d = dev(roi, cuda_device)
    mask_d = dev(mask.view(np.uint8) * np.uint8(255), cuda_device)
    mask_t_d = dev(mask_t, cuda_device)
    got = ops.roi_median(roi_d, mask_d, mask_t=mask_t_d).cpu().numpy()
    assert ops.last_gather_path().median_npt == median_npt(L)
    np.testing.assert_array_equal(got, want)
    stats = torch.full(roi.shape[:3] + (ops.NSTATS,), -7.0, dtype=torch.float64, device=cuda_device)
    ops._median_into(roi_d, mask_d, mask_t_d, tm, stats, 6)
    s = stats.cpu().numpy()
    np.testing.assert_array_equal(s[..., 6], want)
    assert (s[..., [0, 1, 2, 3, 4, 5, 7]] == -7.0).all()
    if dtype == np.float32 and L * L >= 4:
        # windows (c, t) of markers 2 and 3 hold the F32_SPECIAL values in this order
        assert got[2, 0, 0] == 1.0 and got[2, 0, 1] == np.inf and got[2, 0, 2] == 0.0
        assert np.isnan(got[2, 1, 0]) and got[2, 1, 1] == 5.0 and got[2, 1, 2] == -1.25
        assert got[3, 0, 0] == 0.0 and got[3, 0, 1] == -np.inf and got[3, 1, 0] == 0.5
        assert got[3, 1, 1] == -np.inf and got[3, 1, 2] == 2.0 ** -148   # 1.5 x 2^-149, rounded to even
    assert np.isnan(got[5]).all()


@gpu
@pytest.mark.parametrize("L", [16, 17, 34, 35, 72])
@pytest.mark.parametrize("mask_off", [0, 1])
def test_roi_stats_u16_kernels(cuda_device, gather_settings, L, mask_off):
    """roi_stats on uint16 crops reads every marker's block as its own image: the word kernel
    for even L with 2-byte aligned masks, the element kernel for odd L or masks at odd
    addresses; 0/255 mask bytes; counts and sums exact, medians from the separate pass."""
    from magnify_b200 import ops

    m, c, t = 7, 2, 3
    rng = np.random.default_rng(L * 2 + mask_off)
    roi = rng.integers(0, 65535, (m, c, t, L, L), dtype=np.uint16, endpoint=True)
    roi[:, 1] = 65535
    fg = rng.random((m, 2, L, L)) < 0.4
    bg = ~fg
    fg[3] = False
    mask_t = np.array([0, 1, 1], dtype=np.int32)
    case = _case(L=L, M=m, mask_off=mask_off, values="saturated")
    fg_d, bg_d = _mask_bytes(case, rng, fg, cuda_device), _mask_bytes(case, rng, bg, cuda_device)
    stats = ops.roi_stats(dev(roi, cuda_device), fg_d, bg_d, mask_t=dev(mask_t, cuda_device)).cpu().numpy()
    words = L % 2 == 0 and L > 2 and mask_off % 2 == 0
    path = ops.last_gather_path()
    assert path[:8] == Path("plain-words" if words else "plain-scalar", 0, "word" if words else "element",
                            PLAIN_WARPS, 0, None, True, False)
    assert path.median_npt == median_npt(L)
    fused._check_stats(stats, o_red.masked_stats(roi, fg[:, mask_t], bg[:, mask_t]))


@gpu
@pytest.mark.parametrize("L", [1, 9, 33, 72])
def test_roi_stats_f32(cuda_device, L):
    """roi_stats on float32 crops: NaN pixels of either sign skipped, empty masks NaN, sums in
    float64 against NumPy's float64 sums (rtol 1e-12), medians as np.nanmedian of float32."""
    from magnify_b200 import ops

    m, c, t = 6, 2, 2
    rng = np.random.default_rng(L)
    roi = (rng.standard_normal((m, c, t, L, L)) * 1e4).astype(np.float32)
    nan_px = rng.random(roi.shape) < 0.1
    roi[nan_px] = np.where(rng.random(nan_px.sum()) < 0.5, np.float32(np.nan), -np.float32(np.nan))
    roi[2] = np.nan
    fg = rng.random((m, 1, L, L)) < 0.5
    bg = rng.random((m, 1, L, L)) < 0.7
    fg[1] = False
    stats = ops.roi_stats(dev(roi, cuda_device), dev(fg.view(np.uint8), cuda_device),
                          dev(bg.view(np.uint8), cuda_device)).cpu().numpy()
    r64 = roi.astype(np.float64)
    for k, mask in enumerate((fg, bg)):
        mk = np.broadcast_to(mask[:, None], r64.shape) & ~np.isnan(r64)
        n = mk.sum((-1, -2)).astype(np.float64)
        s = np.where(mk, r64, 0.0).sum((-1, -2))
        np.testing.assert_array_equal(stats[..., k], n)
        np.testing.assert_allclose(stats[..., 2 + k], s, rtol=1e-12, atol=1e-6)
        with np.errstate(invalid="ignore", divide="ignore"):
            np.testing.assert_allclose(stats[..., 4 + k], s / n, rtol=1e-12, atol=1e-9, equal_nan=True)
        np.testing.assert_array_equal(stats[..., 6 + k], o_red.masked_median(roi, mask[:, [0] * t]))
    assert np.isnan(stats[1][..., [4, 6]]).all() and np.isnan(stats[2][..., 4:]).all()
